// dspb200 -- Welch / periodogram / STFT / spectrogram.
//
// Reference path: src/periodograms.jl -- ArraySplit (:32-73), fft2pow! (:142-172), fft2oneortwosided!
// (:234-244), welch_pgram_helper! (:746-759), stft (:872-897).
//
// Fused path (power-of-two nfft that fits shared memory): one kernel does segment gather, window
// multiply (Float64 product rounded to the signal eltype, :66), the FFT out of shared memory and
//   * Welch: |Z|^2 accumulated in registers across all segments a CTA owns; real signals ride two
//     segments per complex FFT (z = a + i b), and because |A_k|^2 + |B_k|^2 = (|Z_k|^2 + |Z_{N-k}|^2)/2
//     the split is deferred to the finalize kernel -- the inner loop never un-mixes the two spectra.
//   * STFT / spectrogram: the spectrum is parked in shared memory (natural order), un-mixed per bin and
//     stored column by column, coalesced along frequency.
// Generic path (any other nfft): segment/window kernel -> batched cuFFT -> power / store kernels.
#include "fft_core.cuh"
#include "fft_r32.cuh"
#include "async_copy.cuh"
#include <cufft.h>
#include <math.h>
#include <new>
#include <vector>

namespace dspb200 {

struct SpecPlanImpl {
    int dtype = 0;
    bool cplx = false, f64 = false;
    int64_t n = 0, noverlap = 0, hop = 0, nfft = 0;
    int onesided = 0;
    int64_t nout = 0;
    bool fused = false;
    int device = 0;
    int sm_count = 148;
    void* d_window = nullptr;     // n window values (double, or float2 hi/lo pairs for Float32 signals) or null
    void* d_tw = nullptr;         // last-pass twiddle table (fused; fft_fill_tl)
    void* d_t32 = nullptr;        // nfft = 1024, Float32: W_1024^t rows of the warp-per-unit STFT kernel (stft_w1k_kernel)
    void* d_t16 = nullptr;        // cx<T>[16][8], cx<T>[256][8]: radix-16 twiddle tables (fused)
    void* d_t256 = nullptr;
    size_t smem_optin = 0;        // cudaDevAttrMaxSharedMemoryPerBlockOptin
    int64_t ntapers = 0;          // multitaper plans: d_window holds ntapers rows of n values
    DevBuf tmp;                   // multitaper spectrogram: one taper's PSD matrix
    // launch configuration of the fused Welch kernel, chosen once per (plan, alignment class): the selection walks up to nine
    // kernel instances through cudaFuncSetAttribute + the occupancy calculator (tens of microseconds per launch otherwise)
    struct WelchCfg { void* kern = nullptr; size_t smem = 0; int g = 0, per_sm = 0, threads = 0; };
    WelchCfg welch_cfg[2];        // [0]: unaligned segments (direct loads), [1]: TMA-capable
    int nparts = 0;               // CTAs of the Welch kernel == rows of `partial`
    int rows_used = 0;            // rows of `partial` written since welch_begin (host bookkeeping, stream order = call order)
    DevBuf partial;               // fused Welch: [nparts][nfft] real T
    // generic path
    cufftHandle fft = 0;
    bool fft_ok = false;
    int64_t batch = 0;            // segments per cuFFT call
    int64_t nbins_fft = 0;        // nfft/2+1 (real) or nfft (complex)
    DevBuf segbuf, specbuf, acc;  // acc: double[nbins_fft]
    // host-pointer path
    DevBuf in[2], out;
    cudaStream_t s_copy = nullptr, s_exec = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
};

// ---------------------------------------------------------------------------------------------- helpers
// src/periodograms.jl:66 forms sample * window in Float64 (window functions return Vector{Float64}) and rounds
// the product to the buffer eltype.  Float64 signals: one DMUL.  Float32 signals: the window is held as an
// unevaluated float pair w = wh + wl (|wl| <= ulp(wh)/2) and the product is fma(x, wh, x*wl): it equals
// round(x * w * (1 + e)), |e| < 2^-47, i.e. the reference's correctly rounded value except when x*w falls within
// 2^-47 (relative) of a Float32 rounding boundary (about one sample in 10^7, then off by one ulp) -- without
// putting two conversions and a DMUL per sample on the FP64 pipe.
template <typename T> struct win_t { using type = double; };
template <> struct win_t<float> { using type = float2; };
__device__ __forceinline__ double win_mul(double v, double w) { return v * w; }
__device__ __forceinline__ float win_mul(float v, float2 w) { return fmaf(v, w.x, v * w.y); }

template <typename T, bool CPLX> struct in_type { using type = T; };
template <typename T> struct in_type<T, true> { using type = cx<T>; };

// ---------------------------------------------------------------------------------------------- fused Welch
// Persistent CTAs; CTA c owns a contiguous range of units (unit = one complex segment, or two consecutive real
// segments packed as re/im).  TMA variant: the raw samples of the NEXT unit (one contiguous hop+n range) are
// fetched by a single cp.async.bulk into a staging buffer while the current unit's FFT passes run, so the HBM
// latency of the segment loads is off the critical path; the first FFT pass reads the staged samples from
// shared memory.  The direct variant (unaligned segments, or staging does not fit) loads from global memory
// in the first pass.
// MODE 0: direct loads; 1: TMA staging; 2: TMA staging + the window table copied to shared memory once per CTA (when
// that does not cost residency): the per-unit window reads were the kernel's main long-scoreboard stall;
// 3: TMA staging + the window in REGISTERS: thread t multiplies the samples j = t + r N/16 of every segment, so its 16
// window values never change -- they are loaded once (32 registers for the Float32 hi/lo pairs), which removes the window
// reads (13 % of the kernel's shared-memory wavefronts at nfft = 4096) and the 32 KB table.
// G > 1: G independent thread groups per CTA, each a "virtual CTA" with its own data buffer, staging buffer and mbarrier
// and its own range of units, synchronising among themselves only (named barriers); the groups share ONE copy of the
// twiddle tables and of the window table, so three 4096-point transforms fit one SM where two single-group CTAs with
// private tables did (ncu on the two-CTA configuration: 4 warps per scheduler, issue slots 60 % busy, the stalls that
// remain -- wait, short scoreboard -- are latency a third warp set hides).
// Shared-memory layout: [tables][window (MODE 2)] then per group [data buffer][staging][mbarrier].
template <typename T, int N, bool CPLX, int MODE> struct welch_layout {
    using In = typename in_type<T, CPLX>::type;
    using W = typename win_t<T>::type;
    __host__ __device__ static size_t table_bytes() { return (size_t)fft_table_elems<T, N>() * sizeof(cx<T>); }
    __host__ __device__ static size_t window_bytes(int64_t n) { return MODE == 2 ? (size_t)n * sizeof(W) : 0; }
    __host__ __device__ static size_t stage_elems(int64_t n, int64_t hop) { return MODE >= 1 ? (size_t)(CPLX ? n : hop + n) : 0; }
    __host__ __device__ static size_t group_bytes(int64_t n, int64_t hop) {
        return (((size_t)padded_len<T>(N) * sizeof(cx<T>) + stage_elems(n, hop) * sizeof(In) + 15) & ~(size_t)15) + 16;
    }
    __host__ __device__ static size_t total(int64_t n, int64_t hop, int groups) {
        return table_bytes() + window_bytes(n) + (size_t)groups * group_bytes(n, hop);
    }
};
template <typename T, int N, int G> struct welch_bounds {
    static constexpr int NTG = fft_threads<N>::value;
    static constexpr int minblocks = G == 1 ? fft_minblocks<T, N>::value : 1;
};

template <typename T, int N, bool CPLX, int MODE, int G>
__global__ void __launch_bounds__((welch_bounds<T, N, G>::NTG * G), (welch_bounds<T, N, G>::minblocks))
welch_fused_kernel(const void* __restrict__ s_, int64_t seg0, int64_t nseg, int64_t hop, int n,
                   int64_t sample_offset, const typename win_t<T>::type* __restrict__ win, const cx<T>* __restrict__ tw,
                   const cx<T>* __restrict__ g16, const cx<T>* __restrict__ g256, T* __restrict__ partial, int fresh_from) {
    constexpr int NT = fft_threads<N>::value;                 // threads of one group
    constexpr int NB16 = N / 16;
    constexpr int ITL = (NB16 + NT - 1) / NT;
    using L = welch_layout<T, N, CPLX, MODE>;
    using Scope = typename std::conditional<G == 1, FftCtaScope, FftGroupScope<NT>>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using In = typename in_type<T, CPLX>::type;
    const In* s = reinterpret_cast<const In*>(s_);
    const int gid = G == 1 ? 0 : threadIdx.x / NT;
    const int tid = G == 1 ? threadIdx.x : threadIdx.x - gid * NT;
    constexpr bool TMA = MODE >= 1;
    constexpr bool WSM = MODE == 2;
    constexpr bool WREG = MODE == 3;
    using W = typename win_t<T>::type;
    cx<T>* tabs = reinterpret_cast<cx<T>*>(smem_raw);
    W* wsm = reinterpret_cast<W*>(smem_raw + L::table_bytes());
    unsigned char* gbase = smem_raw + L::table_bytes() + L::window_bytes(n) + (size_t)gid * L::group_bytes(n, hop);
    cx<T>* sm = reinterpret_cast<cx<T>*>(gbase);
    In* stage = reinterpret_cast<In*>(sm + padded_len<T>(N));                  // TMA staging: hop + n samples
    uint64_t* bar = reinterpret_cast<uint64_t*>(gbase + L::group_bytes(n, hop) - 16);
    // tables and window: staged once by all threads of the CTA
    pdl_launch_dependents();
    const FftCtx<T> ctx = fft_make_ctx_at<T, N, NT * G>(sm, tabs, g16, g256, tw, threadIdx.x);
    if constexpr (WSM) {
        for (int i = threadIdx.x; i < n; i += NT * G) wsm[i] = win[i];
    }
    Scope scope;
    if constexpr (G > 1) scope.id = 8 + gid;
    W wreg[WREG ? ITL : 1][WREG ? 16 : 1];
    if constexpr (WREG) {
#pragma unroll
        for (int it = 0; it < ITL; ++it)
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int j = tid + it * NT + r * NB16;
                wreg[it][r] = (j < n && tid + it * NT < NB16) ? win[j] : W{};
            }
    }

    T acc[ITL][16];                                   // thread t: |X[t + it NT + r N/16]|^2 summed over its units (natural order)
#pragma unroll
    for (int i = 0; i < ITL; ++i)
#pragma unroll
        for (int r = 0; r < 16; ++r) acc[i][r] = T(0);

    const int64_t units = CPLX ? nseg : (nseg + 1) / 2;
    const int64_t vcta = (int64_t)blockIdx.x * G + gid, nvcta = (int64_t)gridDim.x * G;     // (CTA, group) = virtual CTA
    const int64_t per = (units + nvcta - 1) / nvcta;
    const int64_t u0 = vcta * per < units ? vcta * per : units;
    const int64_t u1 = u0 + per < units ? u0 + per : units;

    auto unit_src = [&](int64_t u) -> const In* { return s + ((seg0 + (CPLX ? u : 2 * u)) * hop - sample_offset); };
    auto unit_bytes = [&](int64_t u) -> uint32_t {
        const bool hasB = !CPLX && (2 * u + 1 < nseg);
        return (uint32_t)((hasB ? hop + n : n) * sizeof(In));
    };
    if constexpr (TMA) {
        if (tid == 0) {
            mbar_init(bar, 1);
            mbar_fence_init();
        }
    }
    pdl_wait();                                       // constants staged; the samples and `partial` come from preceding kernels
    __syncthreads();                                  // twiddle tables staged, barrier initialised
    if constexpr (TMA) {
        if (tid == 0 && u0 < u1) {
            mbar_expect_tx(bar, unit_bytes(u0));
            tma_load_1d(stage, unit_src(u0), unit_bytes(u0), bar);
        }
    }
    uint32_t parity = 0;

    for (int64_t u = u0; u < u1; ++u) {
        const bool hasB = !CPLX && (2 * u + 1 < nseg);
        const In* pa = TMA ? stage : unit_src(u);
        const In* pb = pa + hop;
        if constexpr (TMA) {
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        auto ld0 = [&](int j, int it, int r) -> cx<T> {
            if (j >= n) return mkc<T>(T(0), T(0));
            if constexpr (CPLX) {
                cx<T> v = pa[j];
                if (WREG || WSM || win) { const W w = WREG ? wreg[WREG ? it : 0][WREG ? r : 0] : (WSM ? wsm[j] : win[j]); v = mkc<T>(win_mul(v.x, w), win_mul(v.y, w)); }
                return v;
            } else {
                T a = pa[j];
                T b = hasB ? pb[j] : T(0);
                if (WREG || WSM || win) { const W w = WREG ? wreg[WREG ? it : 0][WREG ? r : 0] : (WSM ? wsm[j] : win[j]); a = win_mul(a, w); b = win_mul(b, w); }
                return mkc<T>(a, b);
            }
        };
        // first pass: the staged samples are read and transformed, then -- one barrier later, which also ends the
        // previous unit's last pass -- stored; once every thread is past its reads the staging buffer is refilled with
        // the next unit while the remaining passes run
        fft_first_pass<T, N, NT, true>(ctx, tid, ld0, scope);
        if constexpr (TMA) {
            if (tid == 0 && u + 1 < u1) {
                mbar_expect_tx(bar, unit_bytes(u + 1));
                tma_load_1d(stage, unit_src(u + 1), unit_bytes(u + 1), bar);
            }
        }
        scope.sync();
        fft_middle<T, N, NT>(ctx, tid, scope);
#pragma unroll
        for (int it = 0; it < ITL; ++it) {
            const int tp = tid + it * NT;
            if (NB16 % NT != 0 && tp >= NB16) break;
            cx<T> v[16];
            fft_last_pass<T, N>(ctx, tp, v);
#pragma unroll
            for (int r = 0; r < 16; ++r) acc[it][r] += cabs2(v[r]);
        }
    }

    // rows below `fresh_from` hold the sums of earlier launches since welch_begin and are added to; the others are
    // written for the first time (no memset of the partial rows, and the finalize pass reads only rows that were written)
    T* dst = partial + vcta * N;
    const bool add = vcta < fresh_from;
#pragma unroll
    for (int it = 0; it < ITL; ++it) {
        const int tp = tid + it * NT;
        if (tp < NB16) {
#pragma unroll
            for (int r = 0; r < 16; ++r) {                                       // natural order, coalesced along tp
                T* q = dst + tp + r * NB16;
                *q = add ? *q + acc[it][r] : acc[it][r];
            }
        }
    }
}

// Reduce the partial spectra that were written since welch_begin (rows < nparts) in Float64, fold the two-for-one mixing
// for real input, apply the fft2pow! scale (m1 = 1/r, m2 = 2/r; :142-172).  A CTA owns 32 consecutive bins; warp s sums
// rows s, s+32, ... (a warp reads 128 contiguous bytes of a row -- the earlier one-warp-per-bin form read a 32-byte sector
// per element and took 14 us for 592 rows, 5 % of the whole C3 Welch), then the 32 slices are added in a fixed order.
template <typename T, int N>
__global__ void __launch_bounds__(1024) welch_finalize_kernel(const T* __restrict__ partial, int nparts, T* __restrict__ out,
                                                              int nout, int real_in, int onesided, double m1, double m2) {
    __shared__ double red[32][33];
    pdl_launch_dependents();
    pdl_wait();
    const int b = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + b;
    double sum = 0.0;
    if (k < nout) {
        const T* c0 = partial + k;                          // the partial spectra are in natural order
        const T* c1 = partial + ((N - k) & (N - 1));
        if (real_in) {
#pragma unroll 4
            for (int c = sl; c < nparts; c += 32) sum += (double)c0[(int64_t)c * N] + (double)c1[(int64_t)c * N];
        } else {
#pragma unroll 4
            for (int c = sl; c < nparts; c += 32) sum += (double)c0[(int64_t)c * N];
        }
    }
    red[sl][b] = sum;
    __syncthreads();
    if (sl == 0 && k < nout) {
#pragma unroll
        for (int i = 1; i < 32; ++i) sum += red[i][b];
        double m = m1;
        if (real_in) {
            sum *= 0.5;
            if (onesided && !(k == 0 || k == N / 2)) m = m2;
        }
        out[k] = (T)(sum * m);
    }
}

// ---------------------------------------------------------------------------------------------- fused STFT
// Persistent CTAs over units (unit = one complex segment or two consecutive real segments of one channel); same
// front end as the Welch kernel (TMA bulk prefetch of the next unit's samples when segment starts are 16-byte
// aligned).  The last pass writes the spectrum back to shared memory in natural order (in place: a thread stores the
// slots it loaded); every thread then emits the bins k = tid + NT*i, un-mixing the two real segments per bin, and the
// global stores of a column are coalesced along frequency.
// MODE 1: PSD columns (fft2pow!), 0: raw spectra (fft2oneortwosided!).  HASB: the unit carries a second real segment
// (-1: decided at run time by `hasB`).  ONES (real input): one-sided output, nout = N/2 + 1 (-1: run time).
template <typename T, int N, bool CPLX, int MODE, int HASB, int ONES, bool ACC = false>
__device__ __forceinline__ void stft_emit(const cx<T>* __restrict__ sm, void* __restrict__ out_, int64_t colA, int nout,
                                          bool hasB_rt, int onesided_rt, T m1, T m2, int tid) {
    constexpr int NT = fft_threads<N>::value;
    // ACC: PSD columns are ADDED to what `out` holds (multitaper spectrogram: one launch per taper, no separate add pass).
    // Compile time: as a run-time predicate the read-modify-write put a scoreboard wait in front of every store (ncu).
    auto put = [&](T* ptr, T val) { if constexpr (ACC) *ptr = *ptr + val; else *ptr = val; };
    const bool hasB = HASB < 0 ? hasB_rt : (HASB != 0);
    const bool onesided = ONES < 0 ? (onesided_rt != 0) : (ONES != 0);
    // `edge`: the bin is DC or Nyquist (scaled by m1 even in a one-sided PSD, src/periodograms.jl:142-172)
    auto emit = [&](int kk, cx<T> zk, cx<T> zm, bool edge) {
        if constexpr (MODE == 1) {                       // PSD columns
            T* out = reinterpret_cast<T*>(out_);
            if constexpr (CPLX) {
                put(out + colA + kk, cabs2(zk) * m1);
            } else {
                // A = (zk + conj zm) / 2, B = (zk - conj zm) / 2i: the halving is exact, so |A|^2 m is formed as the reference does
                const cx<T> A = mkc<T>(T(0.5) * (zk.x + zm.x), T(0.5) * (zk.y - zm.y));
                const cx<T> B = mkc<T>(T(0.5) * (zk.y + zm.y), T(0.5) * (zm.x - zk.x));
                const T m = (onesided && !edge) ? m2 : m1;
                put(out + colA + kk, cabs2(A) * m);
                if (hasB) put(out + colA + nout + kk, cabs2(B) * m);
            }
        } else {                                         // raw spectra
            cx<T>* out = reinterpret_cast<cx<T>*>(out_);
            if constexpr (CPLX) {
                out[colA + kk] = zk;
            } else {
                out[colA + kk] = mkc<T>(T(0.5) * (zk.x + zm.x), T(0.5) * (zk.y - zm.y));
                if (hasB) out[colA + nout + kk] = mkc<T>(T(0.5) * (zk.y + zm.y), T(0.5) * (zm.x - zk.x));
            }
        }
    };
    // the spectrum is in natural order: consecutive lanes read consecutive slots (k) / consecutive slots backwards (N - k)
    if constexpr (NT * 16 == N) {
        // bins kk = tid + Q i: padaddr(kk) = padaddr(tid) + padaddr(Q i), and for tid > 0
        // padaddr(N - kk) = padaddr(Q - tid) + padaddr(Q (15 - i)) -- every per-bin offset is a compile-time constant
        // (ncu on the 1024-point spectrogram kernel: a generic loop spent ~50 instructions per output bin, mostly integer
        // address arithmetic and predicates)
        constexpr int Q = N / 16;
        const cx<T>* pk = sm + padaddr<T, N>(tid);
        const cx<T>* pm = tid ? sm + padaddr<T, N>(Q - tid) : sm;
        const bool half = !CPLX && onesided;             // bins 0 .. N/2: i = 0..7 for every thread, bin N/2 for thread 0
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            if (i >= 8 && half) break;
            const cx<T> zk = pk[padaddr<T, N>(Q * i)];
            cx<T> zm = zk;
            if constexpr (!CPLX) zm = pm[tid ? padaddr<T, N>(Q * (15 - i)) : padaddr<T, N>((Q * (16 - i)) & (N - 1))];
            emit(tid + Q * i, zk, zm, (i == 0 || i == 8) && tid == 0);
        }
        if (half && tid == 0) {
            const cx<T> z = sm[padaddr<T, N>(N / 2)];
            emit(N / 2, z, z, true);
        }
    } else {
        for (int kk = tid; kk < nout; kk += NT) {
            const cx<T> zk = sm[padaddr<T, N>(kk)];
            cx<T> zm = zk;
            if constexpr (!CPLX) zm = sm[padaddr<T, N>((N - kk) & (N - 1))];
            emit(kk, zk, zm, kk == 0 || kk == N / 2);
        }
    }
}

// One unit of the STFT kernel.  FAST: n == N (no zero padding) and, for real input, both segments present -- no per-sample
// predicates; WIN: 1 window table present, 0 none (compile time), -1 run time.
template <typename T, int N, bool CPLX, bool TMA, int WIN, bool FAST, class IssueNext>
__device__ __forceinline__ void stft_unit(const FftCtx<T>& ctx, cx<T>* sm, int tid, const typename in_type<T, CPLX>::type* pa,
                                          int64_t hop, int n, bool hasB_rt, const typename win_t<T>::type* __restrict__ win,
                                          void* __restrict__ out_, int64_t colA, int nout, int psd_only, int onesided, T m1,
                                          T m2, IssueNext issue_next) {
    constexpr int NT = fft_threads<N>::value;
    constexpr int NB16 = N / 16;
    constexpr int ITL = (NB16 + NT - 1) / NT;
    using In = typename in_type<T, CPLX>::type;
    const In* pb = pa + hop;
    const bool hasB = FAST ? !CPLX : hasB_rt;
    const bool use_win = WIN < 0 ? (win != nullptr) : (WIN != 0);
    auto ld0 = [&](int j, int, int) -> cx<T> {
        if constexpr (!FAST) { if (j >= n) return mkc<T>(T(0), T(0)); }
        if constexpr (CPLX) {
            cx<T> v = pa[j];
            if (use_win) { const auto w = win[j]; v = mkc<T>(win_mul(v.x, w), win_mul(v.y, w)); }
            return v;
        } else {
            T a = pa[j];
            T b = hasB ? pb[j] : T(0);
            if (use_win) { const auto w = win[j]; a = win_mul(a, w); b = win_mul(b, w); }
            return mkc<T>(a, b);
        }
    };
    // (the barrier inside the first pass also ends the previous unit's emit step)
    fft_first_pass<T, N, NT, true>(ctx, tid, ld0);
    issue_next();                                        // every thread has read the staging buffer: refill it
    __syncthreads();
    fft_middle<T, N, NT>(ctx, tid);
#pragma unroll
    for (int it = 0; it < ITL; ++it) {
        const int tp = tid + it * NT;
        if (NB16 % NT != 0 && tp >= NB16) break;
        cx<T> v[16];
        fft_last_pass<T, N>(ctx, tp, v);
        cx<T>* p = sm + padaddr<T, N>(tp);
#pragma unroll
        for (int r = 0; r < 16; ++r) p[padaddr<T, N>(r * NB16)] = v[r];       // natural order, in place
    }
    __syncthreads();
    constexpr int HB = FAST ? (CPLX ? 0 : 1) : -1;
    if (psd_only & 2) {                                  // bit 1: accumulate into `out` (rare: multitaper)
        stft_emit<T, N, CPLX, 1, -1, -1, true>(sm, out_, colA, nout, hasB, onesided, m1, m2, tid);
    } else if (psd_only) {
        if (CPLX || !onesided) stft_emit<T, N, CPLX, 1, HB, 0>(sm, out_, colA, nout, hasB, 0, m1, m2, tid);
        else stft_emit<T, N, CPLX, 1, HB, 1>(sm, out_, colA, nout, hasB, 1, m1, m2, tid);
    } else {
        stft_emit<T, N, CPLX, 0, HB, -1>(sm, out_, colA, nout, hasB, onesided, m1, m2, tid);
    }
}

// (tried: compiling the Float32 STFT kernels for 768 resident threads per SM -- the 1024-point kernel fits 64 registers and
//  gets 11 CTAs per SM instead of 8 -- C4 1.25 -> 1.40 ms, and the windowed variants spill; kept at 512 threads / 128 registers)
template <typename T, int N, bool CPLX, bool TMA, int WIN>
__global__ void __launch_bounds__(fft_threads<N>::value, fft_minblocks<T, N>::value)
stft_fused_kernel(const void* __restrict__ s_, int64_t chan_stride, int64_t k, int64_t units_per_chan, int64_t total_units,
                  int64_t hop, int n, const typename win_t<T>::type* __restrict__ win, const cx<T>* __restrict__ tw,
                  const cx<T>* __restrict__ g16, const cx<T>* __restrict__ g256, void* __restrict__ out_, int nout,
                  int psd_only, int onesided, T m1, T m2) {
    constexpr int NT = fft_threads<N>::value;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* sm = reinterpret_cast<cx<T>*>(smem_raw);
    using In = typename in_type<T, CPLX>::type;
    const In* s = reinterpret_cast<const In*>(s_);
    const int tid = threadIdx.x;
    const FftCtx<T> ctx = fft_make_ctx<T, N, NT>(sm, g16, g256, tw, tid);
    In* stage = reinterpret_cast<In*>(sm + fft_smem_elems<T, N>());
    uint64_t* bar = reinterpret_cast<uint64_t*>(stage + (CPLX ? n : (hop + n)));

    const int64_t per = (total_units + gridDim.x - 1) / gridDim.x;
    const int64_t u0 = (int64_t)blockIdx.x * per;
    const int64_t u1 = u0 + per < total_units ? u0 + per : total_units;
    // (channel, unit inside the channel) of the current unit, advanced incrementally: no 64-bit division in the loop
    int64_t chan = u0 < u1 ? u0 / units_per_chan : 0;
    int64_t uin = u0 < u1 ? u0 - chan * units_per_chan : 0;
    auto src_of = [&](int64_t c, int64_t u) -> const In* { return s + c * chan_stride + (CPLX ? u : 2 * u) * hop; };
    auto bytes_of = [&](int64_t u) -> uint32_t {
        const bool hb = !CPLX && (2 * u + 1 < k);
        return (uint32_t)((hb ? hop + n : n) * sizeof(In));
    };
    if constexpr (TMA) {
        if (tid == 0) {
            mbar_init(bar, 1);
            mbar_fence_init();
        }
    }
    __syncthreads();
    if constexpr (TMA) {
        if (tid == 0 && u0 < u1) {
            mbar_expect_tx(bar, bytes_of(uin));
            tma_load_1d(stage, src_of(chan, uin), bytes_of(uin), bar);
        }
    }
    uint32_t parity = 0;
    const bool full = (n == N);

    for (int64_t gu = u0; gu < u1; ++gu) {
        const int64_t segA = CPLX ? uin : 2 * uin;
        const bool hasB = !CPLX && (segA + 1 < k);
        const In* pa = TMA ? stage : src_of(chan, uin);
        // the next unit
        int64_t nchan = chan, nuin = uin + 1;
        if (nuin == units_per_chan) { nuin = 0; ++nchan; }
        if constexpr (TMA) {
            mbar_wait(bar, parity);
            parity ^= 1;
        }
        auto issue_next = [&]() {
            if constexpr (TMA) {
                if (tid == 0 && gu + 1 < u1) {
                    mbar_expect_tx(bar, bytes_of(nuin));
                    tma_load_1d(stage, src_of(nchan, nuin), bytes_of(nuin), bar);
                }
            }
        };
        const int64_t colA = (chan * k + segA) * (int64_t)nout;
        if (full && (CPLX || hasB))
            stft_unit<T, N, CPLX, TMA, WIN, true>(ctx, sm, tid, pa, hop, n, hasB, win, out_, colA, nout, psd_only, onesided, m1, m2, issue_next);
        else
            stft_unit<T, N, CPLX, TMA, WIN, false>(ctx, sm, tid, pa, hop, n, hasB, win, out_, colA, nout, psd_only, onesided, m1, m2, issue_next);
        chan = nchan;
        uin = nuin;
    }
}

// ---------------------------------------------------------------------------------------------- 1024-point STFT, one warp per unit
// nfft = 1024 = 32 x 32 (BASELINE config 4): a warp owns a whole transform -- lane c computes the plain 32-point DFT of
// x[c + 32 m], one shared-memory exchange, then lane t the twiddled radix-32 butterfly that leaves X[t + 32 s] -- so a unit
// needs ONE exchange instead of two, no CTA-wide barrier at all (__syncwarp only) and every warp of the SM is an independent
// stream of work (its own staging buffer, mbarrier and TMA prefetch of its next unit).  Float32 only.
namespace w1k {
constexpr int N = 1024;
__host__ __device__ __forceinline__ constexpr int pad(int p) { return p + 2 * (p >> 4) + 2 * (p >> 5); }   // 32-runs 38 apart: odd multiple of 16 B
constexpr int DATA_LEN = 1216;                         // pad(1023) + 1 = 1212, rounded up to a multiple of 4
constexpr int T32_LEN = 32 * 16;
__host__ __device__ inline size_t warp_bytes(int64_t stage_elems, size_t elt) { return (((size_t)DATA_LEN * 8 + (size_t)stage_elems * elt + 15) & ~(size_t)15) + 16; }
}  // namespace w1k

template <bool CPLX, int WIN, int WARPS>
__global__ void __launch_bounds__(32 * WARPS)
stft_w1k_kernel(const void* __restrict__ s_, int64_t chan_stride, int64_t k, int64_t units_per_chan, int64_t total_units,
                int64_t hop, int n, const float2* __restrict__ win, const cx<float>* __restrict__ g32, void* __restrict__ out_,
                int nout, int psd_only, int onesided, float m1, float m2) {
    using T = float;
    using In = typename in_type<T, CPLX>::type;
    constexpr int N = w1k::N;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const In* s = reinterpret_cast<const In*>(s_);
    // layout: [T32][window (n float2, when present)] then per warp [data][staging][mbarrier]
    cx<T>* t32 = reinterpret_cast<cx<T>*>(smem_raw);
    float2* wsm = reinterpret_cast<float2*>(smem_raw + w1k::T32_LEN * sizeof(cx<T>));
    const size_t stage_elems = (size_t)(CPLX ? n : hop + n);
    const size_t wbytes = w1k::warp_bytes((int64_t)stage_elems, sizeof(In));
    unsigned char* wbase = smem_raw + w1k::T32_LEN * sizeof(cx<T>) + (WIN ? (size_t)n * sizeof(float2) : 0) + (size_t)warp * wbytes;
    cx<T>* sm = reinterpret_cast<cx<T>*>(wbase);
    In* stage = reinterpret_cast<In*>(sm + w1k::DATA_LEN);
    uint64_t* bar = reinterpret_cast<uint64_t*>(wbase + wbytes - 16);
    for (int i = threadIdx.x; i < w1k::T32_LEN; i += 32 * WARPS) t32[i] = g32[i];
    if constexpr (WIN != 0) {
        for (int i = threadIdx.x; i < n; i += 32 * WARPS) wsm[i] = win[i];
    }
    if (lane == 0) {
        mbar_init(bar, 1);
        mbar_fence_init();
    }
    __syncthreads();                                    // tables staged, barriers initialised -- the only CTA-wide barrier

    const int64_t vw = (int64_t)blockIdx.x * WARPS + warp, nvw = (int64_t)gridDim.x * WARPS;     // virtual CTA = warp
    const int64_t per = (total_units + nvw - 1) / nvw;
    const int64_t u0 = vw * per < total_units ? vw * per : total_units;
    const int64_t u1 = u0 + per < total_units ? u0 + per : total_units;
    int64_t chan = u0 < u1 ? u0 / units_per_chan : 0;
    int64_t uin = u0 < u1 ? u0 - chan * units_per_chan : 0;
    auto src_of = [&](int64_t c, int64_t u) -> const In* { return s + c * chan_stride + (CPLX ? u : 2 * u) * hop; };
    auto bytes_of = [&](int64_t u) -> uint32_t {
        const bool hb = !CPLX && (2 * u + 1 < k);
        return (uint32_t)((hb ? hop + n : n) * sizeof(In));
    };
    if (lane == 0 && u0 < u1) {
        mbar_expect_tx(bar, bytes_of(uin));
        tma_load_1d(stage, src_of(chan, uin), bytes_of(uin), bar);
    }
    uint32_t parity = 0;
    const bool full = (n == N);
    // twiddle row of this lane's last-pass butterfly (w = W_1024^lane): the same for every unit -- kept in registers
    cx<T> tw[16];
#pragma unroll
    for (int i = 0; i < 16; i += 2) lds2<T>(t32 + ((i >> 1) * 32 + lane) * 2, tw[i], tw[i + 1]);

    for (int64_t gu = u0; gu < u1; ++gu) {
        const int64_t segA = CPLX ? uin : 2 * uin;
        const bool hasB = !CPLX && (segA + 1 < k);
        int64_t nchan = chan, nuin = uin + 1;
        if (nuin == units_per_chan) { nuin = 0; ++nchan; }
        mbar_wait(bar, parity);
        parity ^= 1;
        const In* pa = stage;
        const In* pb = pa + hop;
        // first pass: plain 32-point DFT of x[lane + 32 m] (window applied), 32 contiguous slots at block `lane`
        cx<T> v[32];
        const bool fast = full && (CPLX || hasB);
#pragma unroll
        for (int m = 0; m < 32; ++m) {
            const int j = lane + 32 * m;
            if constexpr (CPLX) {
                cx<T> x = (fast || j < n) ? pa[j] : mkc<T>(0.f, 0.f);
                if constexpr (WIN != 0) { const float2 w = wsm[fast || j < n ? j : 0]; x = mkc<T>(win_mul(x.x, w), win_mul(x.y, w)); }
                v[m] = x;
            } else {
                float a = (fast || j < n) ? pa[j] : 0.f;
                float b = (fast || (hasB && j < n)) ? pb[j] : 0.f;
                if constexpr (WIN != 0) { const float2 w = wsm[fast || j < n ? j : 0]; a = win_mul(a, w); b = win_mul(b, w); }
                v[m] = mkc<T>(a, b);
            }
        }
        __syncwarp();                                   // every lane has read the staging buffer (and the previous unit's spectrum)
        if (lane == 0 && gu + 1 < u1) {                 // refill it with the next unit while this one is transformed
            mbar_expect_tx(bar, bytes_of(nuin));
            tma_load_1d(stage, src_of(nchan, nuin), bytes_of(nuin), bar);
        }
        fft_bfly<T, 32, true>(v, nullptr);
        {
            cx<T>* p = sm + w1k::pad(32 * lane);
#pragma unroll
            for (int r = 0; r < 32; r += 2) sts2<T>(p + w1k::pad(r), v[r], v[r + 1]);
        }
        __syncwarp();
        // last pass: radix 32 at stride 32, twiddles W_1024^lane; the spectrum goes back in natural order, in place
        {
            cx<T>* p = sm + w1k::pad(lane);
#pragma unroll
            for (int r = 0; r < 32; ++r) v[r] = p[38 * r];
            fft_bfly<T, 32, false>(v, tw);
#pragma unroll
            for (int r = 0; r < 32; ++r) p[38 * r] = v[r];
        }
        __syncwarp();
        // emit: bins kk = lane + 32 i; N - kk = (32 - lane) + 32 (31 - i) for lane > 0
        const int64_t colA = (chan * k + segA) * (int64_t)nout;
        const cx<T>* pk = sm + w1k::pad(lane);
        const cx<T>* pm = lane ? sm + w1k::pad(32 - lane) : sm;
        const bool half = !CPLX && onesided;
        // (the accumulate flag is resolved once per unit: as a run-time predicate inside the stores it put a scoreboard wait
        //  in front of every one of them)
        auto emit_all = [&](auto acc_) {
            constexpr bool ACC = decltype(acc_)::value;
            auto put = [&](T* ptr, T val) { if constexpr (ACC) *ptr = *ptr + val; else *ptr = val; };
            auto emit = [&](int kk, cx<T> zk, cx<T> zm, bool edge) {
                if (psd_only) {
                    T* out = reinterpret_cast<T*>(out_);
                    if constexpr (CPLX) {
                        put(out + colA + kk, cabs2(zk) * m1);
                    } else {
                        const cx<T> A = mkc<T>(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
                        const cx<T> B = mkc<T>(0.5f * (zk.y + zm.y), 0.5f * (zm.x - zk.x));
                        const T m = (onesided && !edge) ? m2 : m1;
                        put(out + colA + kk, cabs2(A) * m);
                        if (hasB) put(out + colA + nout + kk, cabs2(B) * m);
                    }
                } else {
                    cx<T>* out = reinterpret_cast<cx<T>*>(out_);
                    if constexpr (CPLX) {
                        out[colA + kk] = zk;
                    } else {
                        out[colA + kk] = mkc<T>(0.5f * (zk.x + zm.x), 0.5f * (zk.y - zm.y));
                        if (hasB) out[colA + nout + kk] = mkc<T>(0.5f * (zk.y + zm.y), 0.5f * (zm.x - zk.x));
                    }
                }
            };
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (i >= 16 && half) break;
                const cx<T> zk = pk[38 * i];
                cx<T> zm = zk;
                if constexpr (!CPLX) zm = pm[lane ? 38 * (31 - i) : 38 * ((32 - i) & 31)];
                emit(lane + 32 * i, zk, zm, (i == 0 || i == 16) && lane == 0);
            }
            if (half && lane == 0) {
                const cx<T> z = sm[w1k::pad(N / 2)];
                emit(N / 2, z, z, true);
            }
        };
        if (psd_only & 2) emit_all(std::true_type{});
        else emit_all(std::false_type{});
        chan = nchan;
        uin = nuin;
    }
}

// ---------------------------------------------------------------------------------------------- generic kernels
// buf[b][j] = window[j] * s[(seg0+b)*hop + j] (j < n), 0 for n <= j < nfft and for b >= nseg.
template <typename T, bool CPLX>
__global__ void seg_window_kernel(const void* __restrict__ s_, int64_t first_sample, int64_t hop, int64_t n,
                                  int64_t nfft, int64_t nseg, int64_t batch, const typename win_t<T>::type* __restrict__ win,
                                  void* __restrict__ buf_) {
    using In = typename in_type<T, CPLX>::type;
    const In* s = reinterpret_cast<const In*>(s_);
    In* buf = reinterpret_cast<In*>(buf_);
    const int64_t total = batch * nfft;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / nfft, j = i - b * nfft;
        In v;
        if constexpr (CPLX) v = mkc<T>(T(0), T(0)); else v = T(0);
        if (b < nseg && j < n) {
            v = s[first_sample + b * hop + j];
            if (win) {
                const auto w = win[j];
                if constexpr (CPLX) v = mkc<T>(win_mul(v.x, w), win_mul(v.y, w)); else v = win_mul(v, w);
            }
        }
        buf[i] = v;
    }
}

// acc[k] += sum_b |X[b][k]|^2  (thread per bin, coalesced along k)
template <typename T>
__global__ void pow_acc_kernel(const cx<T>* __restrict__ X, int64_t nbins, int64_t nseg, double* __restrict__ acc) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nbins) return;
    double sum = 0.0;
    for (int64_t b = 0; b < nseg; ++b) sum += (double)cabs2(X[b * nbins + k]);
    acc[k] += sum;
}

// out[k] from acc (fft2pow! scaling and the real two-sided mirror, :142-172)
template <typename T>
__global__ void pow_finalize_kernel(const double* __restrict__ acc, int64_t nbins_fft, int64_t nfft, int64_t nout,
                                    int onesided, double m1, double m2, T* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nout) return;
    int64_t src = k;
    if (k >= nbins_fft) src = nfft - k;   // mirror of a real FFT
    double m = m1;
    if (onesided && k != 0 && !(k == nbins_fft - 1 && (nfft % 2 == 0))) m = m2;
    out[k] = (T)(acc[src] * m);
}

// STFT store from a batch of spectra X[b][nbins_fft] into columns of out (nout x k)
template <typename T>
__global__ void stft_store_kernel(const cx<T>* __restrict__ X, int64_t nbins_fft, int64_t nfft, int64_t nout,
                                  int64_t nseg, int psd_only, int onesided, T m1, T m2, void* __restrict__ out_,
                                  int64_t col0) {
    const int64_t total = nseg * nout;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / nout, k = i - b * nout;
        const bool mirrored = k >= nbins_fft;
        const cx<T> z = X[b * nbins_fft + (mirrored ? nfft - k : k)];
        if (psd_only) {
            T m = m1;
            if (onesided && k != 0 && !(k == nbins_fft - 1 && (nfft % 2 == 0))) m = m2;
            reinterpret_cast<T*>(out_)[(col0 + b) * nout + k] = cabs2(z) * m;
        } else {
            reinterpret_cast<cx<T>*>(out_)[(col0 + b) * nout + k] = mirrored ? cconj(z) : z;
        }
    }
}

// out[i] += add[i]
template <typename T>
__global__ void acc_add_kernel(T* __restrict__ out, const T* __restrict__ add, int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) out[i] += add[i];
}

// Multitaper cross spectra (src/multitaper.jl:553-616).
// signal is the reference's n_channels x n_samples matrix (channel index fastest); xs gets one contiguous column per
// channel, minus the channel mean when `demean` (:566-570).  One block per channel.
template <typename T>
__global__ void cs_prep_kernel(const T* __restrict__ signal, int64_t nchan, int64_t n, int demean, T* __restrict__ xs) {
    const int64_t c = blockIdx.x;
    __shared__ double red[32];
    __shared__ T mean_s;
    double acc = 0.0;
    if (demean) {
        for (int64_t i = threadIdx.x; i < n; i += blockDim.x) acc += (double)signal[c + nchan * i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
            mean_s = (T)(t / (double)n);
        }
        __syncthreads();
    }
    const T mu = demean ? mean_s : T(0);
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) xs[i + n * c] = signal[c + nchan * i] - mu;
}

// out[l, m, fi] += c_f * x[f, l] * conj(x[f, m]), f = f_lo + fi; x = spectra of ONE taper (rows pre-scaled by
// 1/sqrt(r_t), so the reference's weight 2/r_t and its 1/sqrt(2) on the DC / Nyquist rows become c_f = 2, or 1 there)
template <typename T>
__global__ void cs_acc_kernel(cx<T>* __restrict__ out, const cx<T>* __restrict__ x, int64_t nout, int64_t nchan, int64_t f_lo,
                              int64_t nf, int nyquist_row, int first) {
    const int64_t total = nf * nchan * nchan;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = i % nchan, m = (i / nchan) % nchan, f = f_lo + i / (nchan * nchan);
        const T c = (f == 0 || (nyquist_row && f == nout - 1)) ? T(1) : T(2);
        const cx<T> a = x[f + l * nout], b = x[f + m * nout];
        const cx<T> v = mkc<T>(c * (a.x * b.x + a.y * b.y), c * (a.y * b.x - a.x * b.y));
        out[i] = first ? v : mkc<T>(out[i].x + v.x, out[i].y + v.y);
    }
}

// coherence_from_cs!, src/multitaper.jl:672-693: |S_lm| / sqrt(real(S_ll * S_mm)) from the lower triangle, unit diagonal
template <typename T>
__global__ void coherence_kernel(T* __restrict__ out, const cx<T>* __restrict__ cs, int64_t nchan, int64_t nf) {
    const int64_t total = nf * nchan * nchan;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t l = i % nchan, m = (i / nchan) % nchan, f = i / (nchan * nchan);
        if (l == m) { out[i] = T(1); continue; }
        const int64_t hi = l > m ? l : m, lo = l > m ? m : l;
        const cx<T>* S = cs + f * nchan * nchan;
        const cx<T> s = S[hi + lo * nchan], d1 = S[hi + hi * nchan], d2 = S[lo + lo * nchan];
        out[i] = sqrt(s.x * s.x + s.y * s.y) / sqrt(d1.x * d2.x - d1.y * d2.y);
    }
}

// 2-D periodogram (src/periodograms.jl:175-232, 473-509).  X is the half spectrum of the zero-padded real matrix,
// (n1/2+1) x n2 column-major (first dimension halved, as rfft does).
// ptype 0: out[i, j] = |X_full[i, j]|^2 * m1 over the full n1 x n2 grid (fft2pow2!), conjugate symmetry for i > n1/2.
template <typename T>
__global__ void per2_full_kernel(const cx<T>* __restrict__ X, int64_t n1, int64_t n2, T m1, T* __restrict__ out) {
    const int64_t h = n1 / 2 + 1, total = n1 * n2;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = idx % n1, j = idx / n1;
        const cx<T> v = i < h ? X[i + h * j] : X[(n1 - i) + h * ((n2 - j) % n2)];
        out[idx] = cabs2(v) * m1;
    }
}
// radial forms (fft2pow2radial!): every half-spectrum bin adds |X|^2 * m to its integer wavenumber ring, m = 1/r on the
// rows i = 1 and (n1 even) i = n1/2+1 that have no mirror image, 2/r elsewhere; rings and ring populations are
// accumulated with atomics in Float64 / Int64 (the reference adds in the signal precision, column by column).
template <typename T>
__global__ void per2_radial_kernel(const cx<T>* __restrict__ X, int64_t n1, int64_t n2, double c1, double c2, double m1, double m2,
                                   int64_t kmax, double* __restrict__ acc, unsigned long long* __restrict__ wc) {
    const int64_t h = n1 / 2 + 1, total = h * n2;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = idx % h, j = idx / h;                      // 0-based
        const int64_t kj1 = j <= n2 / 2 ? j : j - n2;
        const double kj = (double)kj1 * c2, a = c1 * (double)i;
        const int64_t wavenum = (int64_t)rint(sqrt(fma(a, a, kj * kj)));    // round(Int, .), ties to even; 0-based ring
        if (wavenum >= kmax) continue;
        const bool single = (i == 0) || (i == h - 1 && n1 % 2 == 0);
        atomicAdd(&acc[wavenum], (double)cabs2(X[idx]) * (single ? m1 : m2));
        atomicAdd(&wc[wavenum], single ? 1ull : 2ull);
    }
}
template <typename T>
__global__ void per2_radial_finish_kernel(const double* __restrict__ acc, const unsigned long long* __restrict__ wc, int64_t kmax,
                                          int average, T* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < kmax) out[k] = (T)(average ? acc[k] / (double)wc[k] : acc[k]);
}
// zero-padded copy of the n1 x n2 signal into the nfft1 x nfft2 transform buffer
template <typename T>
__global__ void per2_pad_kernel(const T* __restrict__ s, int64_t n1, int64_t n2, T* __restrict__ dst, int64_t f1, int64_t f2) {
    const int64_t total = f1 * f2;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = idx % f1, j = idx / f1;
        dst[idx] = (i < n1 && j < n2) ? s[i + n1 * j] : T(0);
    }
}

// ---------------------------------------------------------------------------------------------- dispatch
#define DSP_FUSED_SIZES(X) X(256) X(512) X(1024) X(2048) X(4096) X(8192) X(16384)

static bool fused_size_ok(int64_t nfft, bool f64) {
    if (nfft < 256 || (nfft & (nfft - 1))) return false;
    return nfft <= (f64 ? 8192 : 16384);
}

template <typename K> static int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) DSP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return DSPB200_OK;
}

// Launch configuration of the fused Welch kernel: MODE (staging / window placement) x G (thread groups per CTA).  Every
// candidate that fits is rated by the warps it keeps resident per SM (occupancy calculator x G); ties go to the window
// in shared memory, then to fewer groups.
template <typename T, int N, bool CPLX>
static int launch_welch_fused(SpecPlanImpl* p, const void* s, int64_t seg0, int64_t nseg, int64_t sample_offset,
                              cudaStream_t st) {
    constexpr int NT = fft_threads<N>::value;
    using In = typename in_type<T, CPLX>::type;
    using W = typename win_t<T>::type;
    using Kern = void (*)(const void*, int64_t, int64_t, int64_t, int, int64_t, const W*, const cx<T>*, const cx<T>*, const cx<T>*, T*, int);
    constexpr bool MULTI = sizeof(T) == 4 && N >= 1024 && N <= 4096;       // sizes that get multi-group variants
    // TMA staging needs 16-byte aligned segment starts and sizes
    const uintptr_t first = (uintptr_t)s + (uintptr_t)((seg0 * p->hop - sample_offset) * (int64_t)sizeof(In));
    const bool aligned = (first % 16 == 0) && ((p->hop * sizeof(In)) % 16 == 0) && ((p->n * sizeof(In)) % 16 == 0);
    const int64_t units = CPLX ? nseg : (nseg + 1) / 2;
    if (units < 1) return DSPB200_OK;
    const W* win = reinterpret_cast<const W*>(p->d_window);
    struct Cand { Kern k; size_t smem; int g, warps, per_sm; };
    Cand best{nullptr, 0, 0, -1, 0};
    SpecPlanImpl::WelchCfg& cached = p->welch_cfg[aligned ? 1 : 0];
    if (cached.kern != nullptr) {
        const int64_t cap = (int64_t)p->sm_count * cached.per_sm;
        const int64_t want = cdiv(units, cached.g);
        const int grid = (int)(want < cap ? want : cap);
        DSP_CUDA(launch_pdl(reinterpret_cast<Kern>(cached.kern), (unsigned)grid, (unsigned)cached.threads, cached.smem, st,
                            s, seg0, nseg, p->hop, (int)p->n, sample_offset, win, reinterpret_cast<const cx<T>*>(p->d_tw),
                            reinterpret_cast<const cx<T>*>(p->d_t16), reinterpret_cast<const cx<T>*>(p->d_t256),
                            reinterpret_cast<T*>(p->partial.p), p->rows_used));
        DSP_LAUNCH_OK();
        if (grid * cached.g > p->rows_used) p->rows_used = grid * cached.g;
        return DSPB200_OK;
    }
    // candidates are offered in order of preference (measured sweep, profiles/r2_welch_cfg_sweep.jsonl); the first one that
    // keeps at least 12 warps resident per SM is taken, otherwise the one with the most resident warps
    auto consider = [&](Kern k, size_t smem, int g) -> int {
        if (best.warps >= 12) return DSPB200_OK;
        if (smem > p->smem_optin) return DSPB200_OK;
        DSP_TRY(set_smem(k, smem));
        int per_sm = 0;
        DSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, NT * g, smem));
        if (per_sm < 1) return DSPB200_OK;
        if ((int64_t)per_sm * g * p->sm_count > p->nparts) per_sm = (int)(p->nparts / ((int64_t)g * p->sm_count));
        if (per_sm < 1) return DSPB200_OK;
        const int warps = per_sm * g * NT / 32;
        if (warps > best.warps) best = Cand{k, smem, g, warps, per_sm};
        return DSPB200_OK;
    };
#define DSP_WELCH_CAND(MODE_, G_)                                                                        \
    DSP_TRY(consider(welch_fused_kernel<T, N, CPLX, MODE_, G_>,                                          \
                     welch_layout<T, N, CPLX, MODE_>::total(p->n, p->hop, G_), G_))
    constexpr bool WREGOK = sizeof(T) == 4 && N <= 4096;           // window in registers: 32 extra registers per thread
    if (aligned) {
        if (win) {
            if constexpr (CPLX) {
                // complex: two CTAs per SM with the window in registers (0.303 ms at 2^26 / nfft 4096), then in shared memory (0.319)
                if constexpr (WREGOK) DSP_WELCH_CAND(3, 1);
                DSP_WELCH_CAND(2, 1);
                if constexpr (MULTI) { DSP_WELCH_CAND(3, 2); DSP_WELCH_CAND(2, 2); }
            } else {
                // real: three thread groups sharing tables + window (0.185 ms), then two (0.195), then two CTAs (0.198)
                if constexpr (MULTI) { DSP_WELCH_CAND(2, 3); DSP_WELCH_CAND(2, 2); }
                DSP_WELCH_CAND(2, 1);
                if constexpr (WREGOK) DSP_WELCH_CAND(3, 1);
            }
        }
        if constexpr (MULTI && !CPLX) DSP_WELCH_CAND(1, 3);
        DSP_WELCH_CAND(1, 1);
        if constexpr (MULTI) DSP_WELCH_CAND(1, 2);
    }
    if (best.k == nullptr) DSP_WELCH_CAND(0, 1);
#undef DSP_WELCH_CAND
    DSP_REQUIRE(best.k != nullptr, "no Welch kernel configuration fits (nfft=%lld)", (long long)p->nfft);
    DSP_TRY(set_smem(best.k, best.smem));              // (the last candidate examined may have left a different limit)
    cached.kern = reinterpret_cast<void*>(best.k); cached.smem = best.smem; cached.g = best.g; cached.per_sm = best.per_sm;
    cached.threads = NT * best.g;
    // one wave of persistent CTAs: exactly the number that is co-resident; (CTAs x groups) never exceeds the rows of `partial`
    const int64_t cap = (int64_t)p->sm_count * best.per_sm;
    const int64_t want = cdiv(units, best.g);
    const int grid = (int)(want < cap ? want : cap);
    DSP_CUDA(launch_pdl(best.k, (unsigned)grid, (unsigned)(NT * best.g), best.smem, st, s, seg0, nseg, p->hop, (int)p->n,
                        sample_offset, win, reinterpret_cast<const cx<T>*>(p->d_tw), reinterpret_cast<const cx<T>*>(p->d_t16),
                        reinterpret_cast<const cx<T>*>(p->d_t256), reinterpret_cast<T*>(p->partial.p), p->rows_used));
    DSP_LAUNCH_OK();
    if (grid * best.g > p->rows_used) p->rows_used = grid * best.g;
    return DSPB200_OK;
}

template <typename T, int N>
static int launch_welch_finalize(SpecPlanImpl* p, double r, void* out, cudaStream_t st) {
    const int threads = 1024;
    const int grid = (int)cdiv(p->nout, 32);
    DSP_CUDA(launch_pdl(welch_finalize_kernel<T, N>, (unsigned)grid, (unsigned)threads, (size_t)0, st,
                        reinterpret_cast<const T*>(p->partial.p), p->rows_used, reinterpret_cast<T*>(out), (int)p->nout,
                        p->cplx ? 0 : 1, (int)p->onesided, 1.0 / r, 2.0 / r));
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

template <typename T, int N, bool CPLX>
static int launch_stft_fused(SpecPlanImpl* p, const void* s, int64_t len, int64_t nchan, int64_t k, double r,
                             int psd_only, void* out, cudaStream_t st) {
    constexpr int NT = fft_threads<N>::value;
    using In = typename in_type<T, CPLX>::type;
    const size_t base = (size_t)fft_smem_elems<T, N>() * sizeof(cx<T>);
    const size_t stage = (size_t)(CPLX ? p->n : p->hop + p->n) * sizeof(In) + 16;
    const bool tma = ((uintptr_t)s % 16 == 0) && ((len * sizeof(In)) % 16 == 0 || nchan == 1) &&
                     ((p->hop * sizeof(In)) % 16 == 0) && ((p->n * sizeof(In)) % 16 == 0) &&
                     (base + stage <= p->smem_optin) && (base + stage <= 100 * 1024 || N >= 8192);   // N >= 8192: one CTA per SM anyway
    const size_t smem = tma ? base + stage : base;
    const int64_t upc = CPLX ? k : (k + 1) / 2;
    const int64_t units = upc * nchan;
    if (units < 1) return DSPB200_OK;
    const auto* w = reinterpret_cast<const typename win_t<T>::type*>(p->d_window);
    if constexpr (sizeof(T) == 4 && N == 1024) {
        // one warp per unit (stft_w1k_kernel): needs the TMA alignment conditions
        const bool aligned = ((uintptr_t)s % 16 == 0) && ((len * sizeof(In)) % 16 == 0 || nchan == 1) &&
                             ((p->hop * sizeof(In)) % 16 == 0) && ((p->n * sizeof(In)) % 16 == 0);
        if (aligned && p->d_t32 != nullptr) {
            constexpr int WARPS = 4;
            const size_t smem1 = (size_t)w1k::T32_LEN * sizeof(cx<float>) + (w ? (size_t)p->n * sizeof(float2) : 0) +
                                 (size_t)WARPS * w1k::warp_bytes(CPLX ? p->n : p->hop + p->n, sizeof(In));
            using K1 = void (*)(const void*, int64_t, int64_t, int64_t, int64_t, int64_t, int, const float2*, const cx<float>*, void*, int,
                                int, int, float, float);
            K1 k1 = w ? (K1)stft_w1k_kernel<CPLX, 1, WARPS> : (K1)stft_w1k_kernel<CPLX, 0, WARPS>;
            if (smem1 <= p->smem_optin) {
                DSP_TRY(set_smem(k1, smem1));
                int per = 1;
                DSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, k1, 32 * WARPS, smem1));
                const int64_t cap1 = (int64_t)p->sm_count * (per < 1 ? 1 : per);
                const int64_t want = cdiv(units, WARPS);
                const unsigned grid1 = (unsigned)(want < cap1 ? want : cap1);
                k1<<<grid1, 32 * WARPS, smem1, st>>>(s, len, k, upc, units, p->hop, (int)p->n, reinterpret_cast<const float2*>(w),
                                                      reinterpret_cast<const cx<float>*>(p->d_t32), out, (int)p->nout, psd_only,
                                                      p->onesided, (float)(1.0 / r), (float)(2.0 / r));
                DSP_LAUNCH_OK();
                return DSPB200_OK;
            }
        }
    }
    const auto* tw = reinterpret_cast<const cx<T>*>(p->d_tw);
    const auto* g16 = reinterpret_cast<const cx<T>*>(p->d_t16);
    const auto* g256 = reinterpret_cast<const cx<T>*>(p->d_t256);
    using Kern = void (*)(const void*, int64_t, int64_t, int64_t, int64_t, int64_t, int, const typename win_t<T>::type*, const cx<T>*,
                          const cx<T>*, const cx<T>*, void*, int, int, int, T, T);
    // window presence is a compile-time property of the Float32 kernels (predicated-off window products still issue)
    constexpr bool SPEC = sizeof(T) == 4;
    Kern kern;
    if constexpr (SPEC) {
        if (tma) kern = w ? (Kern)stft_fused_kernel<T, N, CPLX, true, 1> : (Kern)stft_fused_kernel<T, N, CPLX, true, 0>;
        else kern = w ? (Kern)stft_fused_kernel<T, N, CPLX, false, 1> : (Kern)stft_fused_kernel<T, N, CPLX, false, 0>;
    } else {
        kern = tma ? (Kern)stft_fused_kernel<T, N, CPLX, true, -1> : (Kern)stft_fused_kernel<T, N, CPLX, false, -1>;
    }
    DSP_TRY(set_smem(kern, smem));
    int per_sm = 1;
    DSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, NT, smem));
    const int64_t cap = (int64_t)p->sm_count * (per_sm < 1 ? 1 : per_sm);
    const unsigned grid = (unsigned)(units < cap ? units : cap);
    kern<<<grid, NT, smem, st>>>(s, len, k, upc, units, p->hop, (int)p->n, w, tw, g16, g256, out, (int)p->nout, psd_only,
                                 p->onesided, (T)(1.0 / r), (T)(2.0 / r));
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

template <typename T> static int welch_fused_dispatch(SpecPlanImpl* p, const void* s, int64_t seg0, int64_t nseg,
                                                       int64_t sample_offset, cudaStream_t st) {
    switch (p->nfft) {
#define X(NN)                                                                                               \
    case NN:                                                                                                \
        if constexpr (sizeof(T) == 8 && NN > 8192) break;                                                   \
        else return p->cplx ? launch_welch_fused<T, NN, true>(p, s, seg0, nseg, sample_offset, st)          \
                            : launch_welch_fused<T, NN, false>(p, s, seg0, nseg, sample_offset, st);
        DSP_FUSED_SIZES(X)
#undef X
    }
    set_error("no fused Welch kernel for nfft=%lld", (long long)p->nfft);
    return DSPB200_EUNSUPPORTED;
}
template <typename T> static int welch_finalize_dispatch(SpecPlanImpl* p, double r, void* out, cudaStream_t st) {
    switch (p->nfft) {
#define X(NN) case NN: return launch_welch_finalize<T, NN>(p, r, out, st);
        DSP_FUSED_SIZES(X)
#undef X
    }
    return DSPB200_EUNSUPPORTED;
}
template <typename T> static int stft_fused_dispatch(SpecPlanImpl* p, const void* s, int64_t len, int64_t nchan,
                                                      int64_t k, double r, int psd_only, void* out, cudaStream_t st) {
    switch (p->nfft) {
#define X(NN)                                                                                               \
    case NN:                                                                                                \
        if constexpr (sizeof(T) == 8 && NN > 8192) break;                                                   \
        else return p->cplx ? launch_stft_fused<T, NN, true>(p, s, len, nchan, k, r, psd_only, out, st)     \
                            : launch_stft_fused<T, NN, false>(p, s, len, nchan, k, r, psd_only, out, st);
        DSP_FUSED_SIZES(X)
#undef X
    }
    set_error("no fused STFT kernel for nfft=%lld", (long long)p->nfft);
    return DSPB200_EUNSUPPORTED;
}

// ---------------------------------------------------------------------------------------------- generic path
static int cufft_fail(cufftResult r, const char* what) {
    set_error("cuFFT error %d in %s", (int)r, what);
    return DSPB200_ECUFFT;
}
#define DSP_CUFFT(call)                                          \
    do {                                                         \
        cufftResult r__ = (call);                                \
        if (r__ != CUFFT_SUCCESS) return cufft_fail(r__, #call); \
    } while (0)

static int generic_prepare(SpecPlanImpl* p) {
    if (p->fft_ok) return DSPB200_OK;
    int64_t b = (int64_t(1) << 22) / p->nfft;
    if (b < 1) b = 1;
    if (b > 8192) b = 8192;
    p->batch = b;
    cufftType type = p->cplx ? (p->f64 ? CUFFT_Z2Z : CUFFT_C2C) : (p->f64 ? CUFFT_D2Z : CUFFT_R2C);
    long long nn[1] = {(long long)p->nfft};
    size_t ws = 0;
    DSP_CUFFT(cufftCreate(&p->fft));
    DSP_CUFFT(cufftMakePlanMany64(p->fft, 1, nn, nullptr, 1, 0, nullptr, 1, 0, type, (long long)b, &ws));
    p->fft_ok = true;
    const size_t esz = dtype_size(p->dtype);
    DSP_TRY(p->segbuf.reserve((size_t)(b * p->nfft) * esz));
    DSP_TRY(p->specbuf.reserve((size_t)(b * p->nbins_fft) * (p->f64 ? 16 : 8)));
    DSP_TRY(p->acc.reserve((size_t)p->nbins_fft * sizeof(double)));
    return DSPB200_OK;
}

static int generic_fft(SpecPlanImpl* p, cudaStream_t st) {
    DSP_CUFFT(cufftSetStream(p->fft, st));
    if (p->cplx) {
        if (p->f64) DSP_CUFFT(cufftExecZ2Z(p->fft, (cufftDoubleComplex*)p->segbuf.p, (cufftDoubleComplex*)p->specbuf.p, CUFFT_FORWARD));
        else DSP_CUFFT(cufftExecC2C(p->fft, (cufftComplex*)p->segbuf.p, (cufftComplex*)p->specbuf.p, CUFFT_FORWARD));
    } else {
        if (p->f64) DSP_CUFFT(cufftExecD2Z(p->fft, (cufftDoubleReal*)p->segbuf.p, (cufftDoubleComplex*)p->specbuf.p));
        else DSP_CUFFT(cufftExecR2C(p->fft, (cufftReal*)p->segbuf.p, (cufftComplex*)p->specbuf.p));
    }
    count_launch(1);
    return DSPB200_OK;
}

template <typename T> static int generic_segments(SpecPlanImpl* p, const void* s, int64_t first_sample, int64_t nseg,
                                                   cudaStream_t st) {
    const int64_t total = p->batch * p->nfft;
    const int threads = 256;
    const int grid = (int)(cdiv(total, threads) < 65535 * 8 ? cdiv(total, threads) : 65535 * 8);
    if (p->cplx)
        seg_window_kernel<T, true><<<grid, threads, 0, st>>>(s, first_sample, p->hop, p->n, p->nfft, nseg, p->batch, reinterpret_cast<const typename win_t<T>::type*>(p->d_window), p->segbuf.p);
    else
        seg_window_kernel<T, false><<<grid, threads, 0, st>>>(s, first_sample, p->hop, p->n, p->nfft, nseg, p->batch, reinterpret_cast<const typename win_t<T>::type*>(p->d_window), p->segbuf.p);
    DSP_LAUNCH_OK();
    return generic_fft(p, st);
}

template <typename T> static int welch_generic_acc(SpecPlanImpl* p, const void* s, int64_t sample_offset,
                                                    int64_t seg_begin, int64_t seg_end, cudaStream_t st) {
    for (int64_t b0 = seg_begin; b0 < seg_end; b0 += p->batch) {
        const int64_t nseg = seg_end - b0 < p->batch ? seg_end - b0 : p->batch;
        DSP_TRY(generic_segments<T>(p, s, b0 * p->hop - sample_offset, nseg, st));
        const int threads = 128;
        pow_acc_kernel<T><<<(int)cdiv(p->nbins_fft, threads), threads, 0, st>>>(
            reinterpret_cast<const cx<T>*>(p->specbuf.p), p->nbins_fft, nseg, reinterpret_cast<double*>(p->acc.p));
        DSP_LAUNCH_OK();
    }
    return DSPB200_OK;
}

template <typename T> static int stft_generic(SpecPlanImpl* p, const void* s, int64_t len, int64_t nchan, int64_t k,
                                               double r, int psd_only, void* out, cudaStream_t st) {
    for (int64_t c = 0; c < nchan; ++c) {
        for (int64_t b0 = 0; b0 < k; b0 += p->batch) {
            const int64_t nseg = k - b0 < p->batch ? k - b0 : p->batch;
            DSP_TRY(generic_segments<T>(p, s, c * len + b0 * p->hop, nseg, st));
            const int64_t total = nseg * p->nout;
            const int threads = 256;
            const int grid = (int)(cdiv(total, threads) < 65535 * 8 ? cdiv(total, threads) : 65535 * 8);
            stft_store_kernel<T><<<grid, threads, 0, st>>>(reinterpret_cast<const cx<T>*>(p->specbuf.p), p->nbins_fft,
                                                           p->nfft, p->nout, nseg, psd_only, p->onesided, (T)(1.0 / r),
                                                           (T)(2.0 / r), out, c * k + b0);
            DSP_LAUNCH_OK();
        }
    }
    return DSPB200_OK;
}

// ---------------------------------------------------------------------------------------------- plan-level ops
static int welch_begin(SpecPlanImpl* p, cudaStream_t st) {
    if (p->fused) {
        p->rows_used = 0;            // the first launch writes its rows, later ones add (welch_fused_kernel, `fresh_from`)
    } else {
        DSP_TRY(generic_prepare(p));
        DSP_CUDA(cudaMemsetAsync(p->acc.p, 0, (size_t)p->nbins_fft * sizeof(double), st));
    }
    return DSPB200_OK;
}

static int welch_accumulate(SpecPlanImpl* p, const void* s, int64_t sample_offset, int64_t seg_begin, int64_t seg_end,
                            cudaStream_t st) {
    if (seg_end <= seg_begin) return DSPB200_OK;
    if (p->fused) {
        return p->f64 ? welch_fused_dispatch<double>(p, s, seg_begin, seg_end - seg_begin, sample_offset, st)
                      : welch_fused_dispatch<float>(p, s, seg_begin, seg_end - seg_begin, sample_offset, st);
    }
    return p->f64 ? welch_generic_acc<double>(p, s, sample_offset, seg_begin, seg_end, st)
                  : welch_generic_acc<float>(p, s, sample_offset, seg_begin, seg_end, st);
}

static int welch_finalize(SpecPlanImpl* p, double r, void* out, cudaStream_t st) {
    if (p->fused) return p->f64 ? welch_finalize_dispatch<double>(p, r, out, st) : welch_finalize_dispatch<float>(p, r, out, st);
    const int threads = 128;
    const int grid = (int)cdiv(p->nout, threads);
    if (p->f64)
        pow_finalize_kernel<double><<<grid, threads, 0, st>>>((const double*)p->acc.p, p->nbins_fft, p->nfft, p->nout, p->onesided, 1.0 / r, 2.0 / r, (double*)out);
    else
        pow_finalize_kernel<float><<<grid, threads, 0, st>>>((const double*)p->acc.p, p->nbins_fft, p->nfft, p->nout, p->onesided, 1.0 / r, 2.0 / r, (float*)out);
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

static int64_t nsegments(const SpecPlanImpl* p, int64_t len) {
    return len >= p->n ? (len - p->n) / p->hop + 1 : 0;   // src/periodograms.jl:49-50
}

static int ensure_streams(SpecPlanImpl* p) {
    if (p->s_exec) return DSPB200_OK;
    DSP_CUDA(cudaStreamCreateWithFlags(&p->s_copy, cudaStreamNonBlocking));
    DSP_CUDA(cudaStreamCreateWithFlags(&p->s_exec, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        DSP_CUDA(cudaEventCreateWithFlags(&p->ev_in[i], cudaEventDisableTiming));
        DSP_CUDA(cudaEventCreateWithFlags(&p->ev_done[i], cudaEventDisableTiming));
    }
    return DSPB200_OK;
}

}  // namespace dspb200

using namespace dspb200;

struct dspb200_spec_plan {
    SpecPlanImpl impl;
};

static size_t win_row_bytes(const SpecPlanImpl* p) { return (size_t)p->n * sizeof(double); }   // float2 pairs are 8 B too

// mt_cross_power_spectra! / mt_coherence!, src/multitaper.jl:553-603, 722-790 (host pointers)
template <typename T>
static int mt_cross_run(dspb200_spec_plan* plan, const void* signal, int64_t nchan, int demean, int64_t f_lo, int64_t nf,
                        int coherence, void* out, bool dev = false, cudaStream_t user_stream = 0) {
    SpecPlanImpl* p = &plan->impl;
    cudaStream_t st = dev ? user_stream : p->s_exec;
    const int64_t n = p->n, cnt = nchan * nchan * nf;
    const size_t cs_bytes = (size_t)cnt * sizeof(cx<T>), out_bytes = coherence ? (size_t)cnt * sizeof(T) : cs_bytes;
    if (!dev) DSP_TRY(p->in[0].reserve((size_t)(n * nchan) * sizeof(T)));
    DSP_TRY(p->in[1].reserve((size_t)(n * nchan) * sizeof(T)));
    DSP_TRY(p->tmp.reserve((size_t)(p->nout * nchan) * sizeof(cx<T>)));
    DSP_TRY(p->out.reserve(cs_bytes + (coherence ? out_bytes : 0)));
    if (!dev) DSP_CUDA(cudaMemcpyAsync(p->in[0].p, signal, (size_t)(n * nchan) * sizeof(T), cudaMemcpyHostToDevice, st));
    cs_prep_kernel<T><<<(unsigned)nchan, 256, 0, st>>>(dev ? (const T*)signal : (const T*)p->in[0].p, nchan, n, demean, (T*)p->in[1].p);
    DSP_LAUNCH_OK();
    const int threads = 256;
    const int grid = (int)(cdiv(cnt, threads) < 148 * 32 ? cdiv(cnt, threads) : 148 * 32);
    void* const base = p->d_window;
    int rc = DSPB200_OK;
    for (int64_t t = 0; t < p->ntapers && rc == DSPB200_OK; ++t) {
        p->d_window = (char*)base + (size_t)t * win_row_bytes(p);
        rc = dspb200_stft_exec_dev(plan, p->in[1].p, n, nchan, 1.0, 0, p->tmp.p, st);     // raw spectra, nout x nchan
        if (rc == DSPB200_OK) {
            cs_acc_kernel<T><<<grid, threads, 0, st>>>((cx<T>*)p->out.p, (const cx<T>*)p->tmp.p, p->nout, nchan, f_lo, nf,
                                                       (p->nfft % 2 == 0) ? 1 : 0, t == 0 ? 1 : 0);
            count_launch(1);
        }
    }
    p->d_window = base;
    DSP_TRY(rc);
    void* res = p->out.p;
    if (coherence) {
        res = (char*)p->out.p + cs_bytes;
        coherence_kernel<T><<<grid, threads, 0, st>>>((T*)res, (const cx<T>*)p->out.p, nchan, nf);
        DSP_LAUNCH_OK();
    }
    DSP_CUDA(cudaMemcpyAsync(out, res, out_bytes, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    DSP_CUDA(cudaStreamSynchronize(st));                 // the plan's scratch is reused by the next call
    return DSPB200_OK;
}

template <typename T>
static int periodogram2_run(const void* s, int64_t n1, int64_t n2, int64_t f1, int64_t f2, double r, int ptype, void* out,
                            bool dev = false, cudaStream_t st = 0) {
    const int64_t h = f1 / 2 + 1, nmin = f1 < f2 ? f1 : f2, kmax = nmin / 2 + 1;
    const int64_t nout = ptype == 0 ? f1 * f2 : kmax;
    const int threads = 256;
    auto grid = [&](int64_t total) { const int64_t g = cdiv(total, threads); return (int)(g < 148 * 32 ? g : 148 * 32); };
    ConvenienceLock lock;                                       // cached plan + scratch arena (common.cuh)
    DevBuf &ds = scratch_buf(0), &dpad = scratch_buf(1), &dX = scratch_buf(2), &dout = scratch_buf(3), &dacc = scratch_buf(4);
    cufftHandle plan = 0;
    auto body = [&]() -> int {
        if (!dev) DSP_TRY(ds.reserve((size_t)(n1 * n2) * sizeof(T)));
        DSP_TRY(dpad.reserve((size_t)(f1 * f2) * sizeof(T)));
        DSP_TRY(dX.reserve((size_t)(h * f2) * sizeof(cx<T>)));
        if (!dev) {
            DSP_TRY(dout.reserve((size_t)nout * sizeof(T)));
            DSP_CUDA(cudaMemcpy(ds.p, s, (size_t)(n1 * n2) * sizeof(T), cudaMemcpyHostToDevice));
        }
        const T* src = dev ? (const T*)s : (const T*)ds.p;
        T* dst = dev ? (T*)out : (T*)dout.p;
        per2_pad_kernel<T><<<grid(f1 * f2), threads, 0, st>>>(src, n1, n2, (T*)dpad.p, f1, f2);
        DSP_LAUNCH_OK();
        long long nn[2] = {(long long)f2, (long long)f1};            // cuFFT is row-major: slowest dimension first
        int hp = 0;
        DSP_TRY(plan_cache_get(&hp, 2, nn, false, 0, 0, sizeof(T) == 8 ? CUFFT_D2Z : CUFFT_R2C, 1));
        plan = (cufftHandle)hp;
        DSP_CUFFT(cufftSetStream(plan, st));
        if (sizeof(T) == 8) DSP_CUFFT(cufftExecD2Z(plan, (cufftDoubleReal*)dpad.p, (cufftDoubleComplex*)dX.p));
        else DSP_CUFFT(cufftExecR2C(plan, (cufftReal*)dpad.p, (cufftComplex*)dX.p));
        count_launch(1);
        if (ptype == 0) {
            per2_full_kernel<T><<<grid(f1 * f2), threads, 0, st>>>((const cx<T>*)dX.p, f1, f2, (T)(1.0 / r), dst);
            DSP_LAUNCH_OK();
        } else {
            DSP_TRY(dacc.reserve((size_t)kmax * 16));
            DSP_CUDA(cudaMemsetAsync(dacc.p, 0, (size_t)kmax * 16, st));
            double* acc = (double*)dacc.p;
            unsigned long long* wc = (unsigned long long*)(acc + kmax);
            double c1 = 1.0, c2 = 1.0;                               // wavevector scaling for non-square transforms, :193-199
            if (f1 == nmin) c2 = (double)f1 / (double)f2; else c1 = (double)f2 / (double)f1;
            const T m1 = (T)(1.0 / r), m2 = (T)(2.0 / r);            // rounded to the signal precision as in the reference
            per2_radial_kernel<T><<<grid(h * f2), threads, 0, st>>>((const cx<T>*)dX.p, f1, f2, c1, c2, (double)m1, (double)m2, kmax, acc, wc);
            DSP_LAUNCH_OK();
            per2_radial_finish_kernel<T><<<(unsigned)cdiv(kmax, threads), threads, 0, st>>>(acc, wc, kmax, ptype == 2, dst);
            DSP_LAUNCH_OK();
        }
        if (dev) DSP_CUDA(cudaStreamSynchronize(st));      // the cached plan and the arena are reused by the next call
        else DSP_CUDA(cudaMemcpy(out, dout.p, (size_t)nout * sizeof(T), cudaMemcpyDeviceToHost));
        return DSPB200_OK;
    };
    const int rc = body();
    scratch_trim((size_t)256 << 20);
    return rc;
}

extern "C" {

static int spec_plan_create_impl(dspb200_spec_plan** plan, int dtype, int64_t n, int64_t noverlap, int64_t nfft,
                                 int onesided, const double* window_host, int64_t nrows) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    *plan = nullptr;
    DSP_REQUIRE(dtype_valid(dtype), "invalid dtype %d", dtype);
    DSP_REQUIRE(n >= 1, "n must be >= 1 (got %lld)", (long long)n);
    DSP_REQUIRE(noverlap >= 0 && noverlap < n, "noverlap must be between zero and n");   // DomainError :44
    DSP_REQUIRE(nfft >= n, "nfft must be >= n");                                           // DomainError :45
    DSP_REQUIRE(!(onesided && dtype_is_cplx(dtype)), "cannot compute one-sided FFT of a complex signal");  // :564
    DSP_REQUIRE(nfft < (int64_t(1) << 31), "nfft too large");
    dspb200_spec_plan* h = new (std::nothrow) dspb200_spec_plan();
    DSP_REQUIRE(h != nullptr, "out of host memory");
    SpecPlanImpl* p = &h->impl;
    p->dtype = dtype; p->cplx = dtype_is_cplx(dtype); p->f64 = dtype_is_f64(dtype);
    p->n = n; p->noverlap = noverlap; p->hop = n - noverlap; p->nfft = nfft; p->onesided = onesided ? 1 : 0;
    p->nout = onesided ? nfft / 2 + 1 : nfft;
    p->nbins_fft = p->cplx ? nfft : nfft / 2 + 1;
    p->fused = fused_size_ok(nfft, p->f64);
    int rc = DSPB200_OK;
    do {
        if (cudaGetDevice(&p->device) != cudaSuccess) { rc = cuda_fail(cudaGetLastError(), "cudaGetDevice", __FILE__, __LINE__); break; }
        p->sm_count = device_sm_count();
        if (window_host) {
            const int64_t nw = n * (nrows < 1 ? 1 : nrows);
            p->ntapers = nrows;
            cudaError_t e = cudaMalloc(&p->d_window, (size_t)nw * sizeof(double));
            if (e == cudaSuccess) {
                if (p->f64) {
                    e = cudaMemcpy(p->d_window, window_host, (size_t)nw * sizeof(double), cudaMemcpyHostToDevice);
                } else {                                   // hi/lo float pairs (same 8 bytes per value)
                    std::vector<float> pairs((size_t)nw * 2);
                    for (int64_t j = 0; j < nw; ++j) {
                        const float hi = (float)window_host[j];
                        pairs[2 * j] = hi;
                        pairs[2 * j + 1] = (float)(window_host[j] - (double)hi);
                    }
                    e = cudaMemcpy(p->d_window, pairs.data(), pairs.size() * sizeof(float), cudaMemcpyHostToDevice);
                }
            }
            if (e != cudaSuccess) { rc = cuda_fail(e, "window upload", __FILE__, __LINE__); break; }
        }
        if (p->fused) {
            const size_t csz = p->f64 ? 16 : 8;
            std::vector<unsigned char> tw((size_t)(fft_tl_len_rt(nfft) + 1) * csz), t16((size_t)fft_tw16_len(nfft) * csz), t256((size_t)fft_tw256_len(nfft) * csz);
            if (p->f64) {
                fft_fill_tl<double>((cx<double>*)tw.data(), nfft);
                fft_fill_tables<double>((cx<double>*)t16.data(), (cx<double>*)t256.data(), nfft);
            } else {
                fft_fill_tl<float>((cx<float>*)tw.data(), nfft);
                fft_fill_tables<float>((cx<float>*)t16.data(), (cx<float>*)t256.data(), nfft);
            }
            cudaError_t e = cudaMalloc(&p->d_tw, tw.size());
            if (e == cudaSuccess) e = cudaMemcpy(p->d_tw, tw.data(), tw.size(), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc(&p->d_t16, t16.size());
            if (e == cudaSuccess) e = cudaMemcpy(p->d_t16, t16.data(), t16.size(), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc(&p->d_t256, t256.size());
            if (e == cudaSuccess) e = cudaMemcpy(p->d_t256, t256.data(), t256.size(), cudaMemcpyHostToDevice);
            if (e == cudaSuccess && !p->f64 && nfft == 1024) {                 // table of the warp-per-unit STFT kernel
                std::vector<cx<float>> a32(r32::T32_LEN), a1024(r32::T1024_LEN);
                r32::fill_tables<float>(a32.data(), a1024.data());
                e = cudaMalloc(&p->d_t32, a32.size() * sizeof(cx<float>));
                if (e == cudaSuccess) e = cudaMemcpy(p->d_t32, a32.data(), a32.size() * sizeof(cx<float>), cudaMemcpyHostToDevice);
            }
            int optin = 0;
            if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device);
            p->smem_optin = (size_t)optin;
            if (e != cudaSuccess) { rc = cuda_fail(e, "twiddle upload", __FILE__, __LINE__); break; }
            // persistent Welch grid: CTAs per SM bounded by shared memory (228 KB/SM) and 2048 threads
            // (data + tables + TMA staging for 50 % overlap) per CTA
            const size_t smem = (size_t)(p->f64 ? padded_len<double>((int)nfft) : padded_len<float>((int)nfft)) * csz + (size_t)(fft_tw16_len(nfft) + fft_tw256_len(nfft)) * csz +
                                (size_t)(p->hop + p->n) * (csz / 2);
            int per_sm = (int)((220 * 1024) / (smem + 1024));
            if (per_sm < 4) per_sm = 4;            // up to (CTAs per SM) x (thread groups per CTA) virtual CTAs
            if (per_sm > 8) per_sm = 8;
            p->nparts = p->sm_count * per_sm;      // upper bound; launches use the occupancy API
            rc = p->partial.reserve((size_t)p->nparts * nfft * (p->f64 ? 8 : 4));
            if (rc != DSPB200_OK) break;
        }
    } while (0);
    if (rc != DSPB200_OK) { dspb200_spec_plan_destroy(h); return rc; }
    *plan = h;
    return DSPB200_OK;
}

int dspb200_spec_plan_create(dspb200_spec_plan** plan, int dtype, int64_t n, int64_t noverlap, int64_t nfft,
                             int onesided, const double* window_host) {
    DSP_RANGE("dspb200_spec_plan_create");
    return spec_plan_create_impl(plan, dtype, n, noverlap, nfft, onesided, window_host, 0);
}

int dspb200_mt_plan_create(dspb200_spec_plan** plan, int dtype, int64_t n, int64_t noverlap, int64_t nfft, int onesided,
                           const double* tapers_host, int64_t ntapers) {
    DSP_RANGE("dspb200_mt_plan_create");
    DSP_REQUIRE(tapers_host != nullptr && ntapers >= 1, "tapers must be a non-empty ntapers x n matrix");
    return spec_plan_create_impl(plan, dtype, n, noverlap, nfft, onesided, tapers_host, ntapers);
}

int dspb200_spec_plan_info(const dspb200_spec_plan* plan, int64_t* nout, int* fused) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    if (nout) *nout = plan->impl.nout;
    if (fused) *fused = plan->impl.fused ? 1 : 0;
    return DSPB200_OK;
}

int dspb200_spec_plan_geometry(const dspb200_spec_plan* plan, int* dtype, int64_t* n, int64_t* hop, int64_t* nout) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    if (dtype) *dtype = plan->impl.dtype;
    if (n) *n = plan->impl.n;
    if (hop) *hop = plan->impl.hop;
    if (nout) *nout = plan->impl.nout;
    return DSPB200_OK;
}

int64_t dspb200_spec_nsegments(const dspb200_spec_plan* plan, int64_t len) {
    if (!plan) return -1;
    return nsegments(&plan->impl, len);
}

int dspb200_welch_exec_range_dev(dspb200_spec_plan* plan, const void* s, int64_t len, int64_t sample_offset,
                                 int64_t seg_begin, int64_t seg_end, double r, void* out, void* stream) {
    DSP_RANGE("dspb200_welch_exec_range_dev");
    DSP_REQUIRE(plan && out, "NULL argument");
    DSP_REQUIRE(r != 0.0, "r must be nonzero");
    SpecPlanImpl* p = &plan->impl;
    cudaStream_t st = (cudaStream_t)stream;
    DSP_REQUIRE(seg_begin >= 0 && seg_end >= seg_begin, "bad segment range");
    if (seg_end > seg_begin) {
        DSP_REQUIRE(s != nullptr, "s is NULL");
        DSP_REQUIRE(seg_begin * p->hop >= sample_offset, "segment range starts before the local buffer");
        DSP_REQUIRE((seg_end - 1) * p->hop + p->n <= sample_offset + len, "segment range runs past the local buffer");
    }
    DSP_TRY(welch_begin(p, st));
    DSP_TRY(welch_accumulate(p, s, sample_offset, seg_begin, seg_end, st));
    return welch_finalize(p, r, out, st);
}

// Streaming form of welch_pgram_helper! (src/periodograms.jl:746-759): begin (zero the accumulator), accumulate any number
// of segment ranges -- each from a buffer that holds at least its own samples -- then finalize (fft2pow! scaling).  This is
// what dspb200_welch_exec_range_dev does in one call; the split lets a pipeline feed the segments chunk by chunk.
int dspb200_welch_begin_dev(dspb200_spec_plan* plan, void* stream) {
    DSP_RANGE("dspb200_welch_begin_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    return welch_begin(&plan->impl, (cudaStream_t)stream);
}
int dspb200_welch_accumulate_dev(dspb200_spec_plan* plan, const void* s, int64_t len, int64_t sample_offset,
                                 int64_t seg_begin, int64_t seg_end, void* stream) {
    DSP_RANGE("dspb200_welch_accumulate_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    SpecPlanImpl* p = &plan->impl;
    DSP_REQUIRE(seg_begin >= 0 && seg_end >= seg_begin, "bad segment range");
    if (seg_end == seg_begin) return DSPB200_OK;
    DSP_REQUIRE(s != nullptr, "s is NULL");
    DSP_REQUIRE(seg_begin * p->hop >= sample_offset, "segment range starts before the local buffer");
    DSP_REQUIRE((seg_end - 1) * p->hop + p->n <= sample_offset + len, "segment range runs past the local buffer");
    return welch_accumulate(p, s, sample_offset, seg_begin, seg_end, (cudaStream_t)stream);
}
int dspb200_welch_finalize_dev(dspb200_spec_plan* plan, double r, void* out, void* stream) {
    DSP_RANGE("dspb200_welch_finalize_dev");
    DSP_REQUIRE(plan && out, "NULL argument");
    DSP_REQUIRE(r != 0.0, "r must be nonzero");
    return welch_finalize(&plan->impl, r, out, (cudaStream_t)stream);
}

int dspb200_welch_exec_dev(dspb200_spec_plan* plan, const void* s, int64_t len, double r, void* out, void* stream) {
    DSP_RANGE("dspb200_welch_exec_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    const int64_t k = nsegments(&plan->impl, len);
    return dspb200_welch_exec_range_dev(plan, s, len, 0, 0, k, r, out, stream);
}

// Host-pointer Welch: the signal is streamed through two device buffers in segment-aligned chunks so the
// H2D copy of chunk c+1 overlaps the kernel of chunk c (effective when `s` is pinned).
int dspb200_welch_exec(dspb200_spec_plan* plan, const void* s, int64_t len, double r, void* out) {
    DSP_RANGE("dspb200_welch_exec");
    DSP_REQUIRE(plan && out, "NULL argument");
    DSP_REQUIRE(r != 0.0, "r must be nonzero");
    SpecPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    const size_t esz = dtype_size(p->dtype);
    const int64_t k = nsegments(p, len);
    const size_t out_bytes = (size_t)p->nout * (p->f64 ? 8 : 4);
    DSP_TRY(p->out.reserve(out_bytes));
    DSP_TRY(welch_begin(p, p->s_exec));
    if (k > 0) {
        DSP_REQUIRE(s != nullptr, "s is NULL");
        int64_t chunk_segs = ((int64_t(32) << 20) / (int64_t)esz) / p->hop;   // ~32 MiB of new samples per chunk
        if (chunk_segs < 64) chunk_segs = 64;
        if (chunk_segs > k) chunk_segs = k;
        const size_t chunk_bytes = (size_t)((chunk_segs - 1) * p->hop + p->n) * esz;
        DSP_TRY(p->in[0].reserve(chunk_bytes));
        if (chunk_segs < k) DSP_TRY(p->in[1].reserve(chunk_bytes));
        int slot = 0;
        bool used[2] = {false, false};
        for (int64_t b0 = 0; b0 < k; b0 += chunk_segs, slot ^= 1) {
            const int64_t b1 = b0 + chunk_segs < k ? b0 + chunk_segs : k;
            const int64_t first = b0 * p->hop;
            const int64_t cnt = (b1 - 1 - b0) * p->hop + p->n;
            if (used[slot]) DSP_CUDA(cudaStreamWaitEvent(p->s_copy, p->ev_done[slot], 0));
            DSP_CUDA(cudaMemcpyAsync(p->in[slot].p, (const char*)s + (size_t)first * esz, (size_t)cnt * esz,
                                     cudaMemcpyHostToDevice, p->s_copy));
            DSP_CUDA(cudaEventRecord(p->ev_in[slot], p->s_copy));
            DSP_CUDA(cudaStreamWaitEvent(p->s_exec, p->ev_in[slot], 0));
            DSP_TRY(welch_accumulate(p, p->in[slot].p, first, b0, b1, p->s_exec));
            DSP_CUDA(cudaEventRecord(p->ev_done[slot], p->s_exec));
            used[slot] = true;
        }
    }
    DSP_TRY(welch_finalize(p, r, p->out.p, p->s_exec));
    DSP_CUDA(cudaMemcpyAsync(out, p->out.p, out_bytes, cudaMemcpyDeviceToHost, p->s_exec));
    DSP_CUDA(cudaStreamSynchronize(p->s_exec));
    return DSPB200_OK;
}

// arraysplit / ArraySplit (src/periodograms.jl:32-73, 134-137): all k windowed, zero-padded segments as a k x nfft
// matrix (row = segment; the reference yields them one at a time into a reused buffer).
int dspb200_arraysplit_exec(dspb200_spec_plan* plan, const void* s, int64_t len, void* out) {
    DSP_RANGE("dspb200_arraysplit_exec");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    SpecPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    const int64_t k = nsegments(p, len);
    if (k == 0) return DSPB200_OK;
    DSP_REQUIRE(s && out, "NULL argument");
    const size_t esz = dtype_size(p->dtype);
    const size_t in_bytes = (size_t)len * esz, out_bytes = (size_t)(k * p->nfft) * esz;
    DSP_TRY(p->in[0].reserve(in_bytes));
    DSP_TRY(p->out.reserve(out_bytes));
    DSP_CUDA(cudaMemcpyAsync(p->in[0].p, s, in_bytes, cudaMemcpyHostToDevice, p->s_exec));
    const int64_t total = k * p->nfft;
    const int threads = 256;
    const int grid = (int)(cdiv(total, threads) < 65535 * 8 ? cdiv(total, threads) : 65535 * 8);
#define SEGK(T_, C_) seg_window_kernel<T_, C_><<<grid, threads, 0, p->s_exec>>>(p->in[0].p, 0, p->hop, p->n, p->nfft, k, k, \
        reinterpret_cast<const typename win_t<T_>::type*>(p->d_window), p->out.p)
    if (p->f64) { if (p->cplx) SEGK(double, true); else SEGK(double, false); }
    else { if (p->cplx) SEGK(float, true); else SEGK(float, false); }
#undef SEGK
    DSP_LAUNCH_OK();
    DSP_CUDA(cudaMemcpyAsync(out, p->out.p, out_bytes, cudaMemcpyDeviceToHost, p->s_exec));
    DSP_CUDA(cudaStreamSynchronize(p->s_exec));
    return DSPB200_OK;
}

int dspb200_stft_exec_dev(dspb200_spec_plan* plan, const void* s, int64_t len, int64_t nchan, double r, int psd_only,
                          void* out, void* stream) {
    DSP_RANGE("dspb200_stft_exec_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(r != 0.0 || !psd_only, "r must be nonzero");
    DSP_REQUIRE(nchan >= 0 && len >= 0, "negative size");
    SpecPlanImpl* p = &plan->impl;
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t k = nsegments(p, len);
    if (k == 0 || nchan == 0) return DSPB200_OK;
    DSP_REQUIRE(s && out, "NULL argument");
    if (r == 0.0) r = 1.0;
    if (p->fused)
        return p->f64 ? stft_fused_dispatch<double>(p, s, len, nchan, k, r, psd_only, out, st)
                      : stft_fused_dispatch<float>(p, s, len, nchan, k, r, psd_only, out, st);
    DSP_TRY(generic_prepare(p));
    return p->f64 ? stft_generic<double>(p, s, len, nchan, k, r, psd_only, out, st)
                  : stft_generic<float>(p, s, len, nchan, k, r, psd_only, out, st);
}

int dspb200_stft_exec(dspb200_spec_plan* plan, const void* s, int64_t len, int64_t nchan, double r, int psd_only,
                      void* out) {
    DSP_RANGE("dspb200_stft_exec");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    SpecPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    const int64_t k = nsegments(p, len);
    if (k == 0 || nchan == 0) return DSPB200_OK;
    DSP_REQUIRE(s && out, "NULL argument");
    const size_t esz = dtype_size(p->dtype);
    const size_t in_bytes = (size_t)len * nchan * esz;
    const size_t oel = psd_only ? (p->f64 ? 8 : 4) : (p->f64 ? 16 : 8);
    const size_t out_bytes = (size_t)p->nout * k * nchan * oel;
    DSP_TRY(p->in[0].reserve(in_bytes));
    DSP_TRY(p->out.reserve(out_bytes));
    DSP_CUDA(cudaMemcpyAsync(p->in[0].p, s, in_bytes, cudaMemcpyHostToDevice, p->s_exec));
    DSP_TRY(dspb200_stft_exec_dev(plan, p->in[0].p, len, nchan, r, psd_only, p->out.p, p->s_exec));
    DSP_CUDA(cudaMemcpyAsync(out, p->out.p, out_bytes, cudaMemcpyDeviceToHost, p->s_exec));
    DSP_CUDA(cudaStreamSynchronize(p->s_exec));
    return DSPB200_OK;
}

// Multitaper (SURVEY.md 8f rank 1; src/multitaper.jl:117-242, 262-404).  The plan's window holds `ntapers` rows of n
// samples, each PRE-SCALED by 1/sqrt(r_t) (r_t = fs * sum|w_t|^2 / weight_t, :135-139), so that
//   mt_pgram       = sum_t fft2pow!(FFT(w_t .* s), 1)         (one Welch-style accumulation per taper into one spectrum)
//   mt_spectrogram = sum_t spectrogram(s; window = w_t, r = 1) (one STFT launch per taper + an accumulate kernel)
static int mt_pgram_entry(dspb200_spec_plan* plan, const void* s, int64_t len, void* out, bool dev, cudaStream_t user_stream) {
    DSP_REQUIRE(plan && s && out, "NULL argument");
    SpecPlanImpl* p = &plan->impl;
    DSP_REQUIRE(p->ntapers >= 1, "not a multitaper plan");
    DSP_REQUIRE(len == p->n, "Expected `signal` to be of length `config.n_samples`");          // DimensionMismatch :226
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    cudaStream_t st = dev ? user_stream : p->s_exec;
    const size_t esz = dtype_size(p->dtype);
    const size_t out_bytes = (size_t)p->nout * (p->f64 ? 8 : 4);
    const void* d_s = s;
    if (!dev) {
        DSP_TRY(p->in[0].reserve((size_t)len * esz));
        DSP_TRY(p->out.reserve(out_bytes));
        DSP_CUDA(cudaMemcpyAsync(p->in[0].p, s, (size_t)len * esz, cudaMemcpyHostToDevice, st));
        d_s = p->in[0].p;
    }
    DSP_TRY(welch_begin(p, st));
    void* const base = p->d_window;
    int rc = DSPB200_OK;
    for (int64_t t = 0; t < p->ntapers && rc == DSPB200_OK; ++t) {
        p->d_window = (char*)base + (size_t)t * win_row_bytes(p);
        rc = welch_accumulate(p, d_s, 0, 0, 1, st);
    }
    p->d_window = base;
    DSP_TRY(rc);
    DSP_TRY(welch_finalize(p, 1.0, dev ? out : p->out.p, st));
    if (!dev) DSP_CUDA(cudaMemcpyAsync(out, p->out.p, out_bytes, cudaMemcpyDeviceToHost, st));
    DSP_CUDA(cudaStreamSynchronize(st));
    return DSPB200_OK;
}
int dspb200_mt_pgram_exec(dspb200_spec_plan* plan, const void* s, int64_t len, void* out) {
    DSP_RANGE("dspb200_mt_pgram_exec");
    return mt_pgram_entry(plan, s, len, out, false, 0);
}
int dspb200_mt_pgram_exec_dev(dspb200_spec_plan* plan, const void* d_s, int64_t len, void* d_out, void* stream) {
    DSP_RANGE("dspb200_mt_pgram_exec_dev");
    return mt_pgram_entry(plan, d_s, len, d_out, true, (cudaStream_t)stream);
}

static int mt_spectrogram_entry(dspb200_spec_plan* plan, const void* s, int64_t len, void* out, bool dev, cudaStream_t user_stream) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    SpecPlanImpl* p = &plan->impl;
    DSP_REQUIRE(p->ntapers >= 1, "not a multitaper plan");
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    const int64_t k = nsegments(p, len);
    if (k == 0) return DSPB200_OK;
    DSP_REQUIRE(s && out, "NULL argument");
    cudaStream_t st = dev ? user_stream : p->s_exec;
    const size_t esz = dtype_size(p->dtype), oel = p->f64 ? 8 : 4;
    const int64_t cnt = p->nout * k;
    const void* d_s = s;
    void* d_out = out;
    if (!dev) {
        DSP_TRY(p->in[0].reserve((size_t)len * esz));
        DSP_TRY(p->out.reserve((size_t)cnt * oel));
        DSP_CUDA(cudaMemcpyAsync(p->in[0].p, s, (size_t)len * esz, cudaMemcpyHostToDevice, st));
        d_s = p->in[0].p;
        d_out = p->out.p;
    }
    if (!p->fused) DSP_TRY(p->tmp.reserve((size_t)cnt * oel));
    void* const base = p->d_window;
    int rc = DSPB200_OK;
    for (int64_t t = 0; t < p->ntapers && rc == DSPB200_OK; ++t) {
        p->d_window = (char*)base + (size_t)t * win_row_bytes(p);
        if (p->fused) {                                  // tapers after the first add their PSD columns inside the emit step
            rc = dspb200_stft_exec_dev(plan, d_s, len, 1, 1.0, t == 0 ? 1 : 3, d_out, st);
            continue;
        }
        rc = dspb200_stft_exec_dev(plan, d_s, len, 1, 1.0, 1, t == 0 ? d_out : p->tmp.p, st);
        if (rc == DSPB200_OK && t > 0) {
            const int threads = 256;
            const int grid = (int)(cdiv(cnt, threads) < 148 * 32 ? cdiv(cnt, threads) : 148 * 32);
            if (p->f64) acc_add_kernel<double><<<grid, threads, 0, st>>>((double*)d_out, (const double*)p->tmp.p, cnt);
            else acc_add_kernel<float><<<grid, threads, 0, st>>>((float*)d_out, (const float*)p->tmp.p, cnt);
            count_launch(1);
        }
    }
    p->d_window = base;
    DSP_TRY(rc);
    if (!dev) DSP_CUDA(cudaMemcpyAsync(out, p->out.p, (size_t)cnt * oel, cudaMemcpyDeviceToHost, st));
    DSP_CUDA(cudaStreamSynchronize(st));
    return DSPB200_OK;
}
int dspb200_mt_spectrogram_exec(dspb200_spec_plan* plan, const void* s, int64_t len, void* out) {
    DSP_RANGE("dspb200_mt_spectrogram_exec");
    return mt_spectrogram_entry(plan, s, len, out, false, 0);
}
int dspb200_mt_spectrogram_exec_dev(dspb200_spec_plan* plan, const void* d_s, int64_t len, void* d_out, void* stream) {
    DSP_RANGE("dspb200_mt_spectrogram_exec_dev");
    return mt_spectrogram_entry(plan, d_s, len, d_out, true, (cudaStream_t)stream);
}

static int mt_cross_entry(dspb200_spec_plan* plan, const void* signal, int64_t nchan, int demean, int64_t f_lo, int64_t nf,
                          int coherence, void* out, bool dev, cudaStream_t st) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    SpecPlanImpl* p = &plan->impl;
    DSP_REQUIRE(p->ntapers >= 1, "not a multitaper plan");
    DSP_REQUIRE(!p->cplx && p->onesided,
                "Only real data is supported (with the default choice of `onesided=true`) for this operation.");   // :411-416
    DSP_REQUIRE(nchan >= 1, "n_channels must be positive");
    DSP_REQUIRE(f_lo >= 0 && nf >= 0 && f_lo + nf <= p->nout, "frequency range outside the spectrum");
    if (nf == 0) return DSPB200_OK;
    DSP_REQUIRE(signal && out, "NULL argument");
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    return p->f64 ? mt_cross_run<double>(plan, signal, nchan, demean, f_lo, nf, coherence, out, dev, st)
                  : mt_cross_run<float>(plan, signal, nchan, demean, f_lo, nf, coherence, out, dev, st);
}
int dspb200_mt_cross_spectra_exec(dspb200_spec_plan* plan, const void* signal, int64_t nchan, int demean, int64_t f_lo,
                                  int64_t nf, int coherence, void* out) {
    DSP_RANGE("dspb200_mt_cross_spectra_exec");
    return mt_cross_entry(plan, signal, nchan, demean, f_lo, nf, coherence, out, false, 0);
}
int dspb200_mt_cross_spectra_exec_dev(dspb200_spec_plan* plan, const void* d_signal, int64_t nchan, int demean, int64_t f_lo,
                                      int64_t nf, int coherence, void* d_out, void* stream) {
    DSP_RANGE("dspb200_mt_cross_spectra_exec_dev");
    return mt_cross_entry(plan, d_signal, nchan, demean, f_lo, nf, coherence, d_out, true, (cudaStream_t)stream);
}

// periodogram(s::AbstractMatrix; nfft, fs, radialsum, radialavg), src/periodograms.jl:473-509 (cached plan + scratch arena)
static int periodogram2_entry(int dtype, const void* s, int64_t n1, int64_t n2, int64_t nfft1, int64_t nfft2, double r, int ptype,
                              void* out, bool dev, cudaStream_t st) {
    DSP_REQUIRE(dtype == DSPB200_F32 || dtype == DSPB200_F64, "periodogram of a matrix takes a real signal (dtype %d)", dtype);
    DSP_REQUIRE(s && out, "NULL argument");
    DSP_REQUIRE(n1 > 1 && n2 > 1, "dimensions of s must be > 1");                                   // :478
    DSP_REQUIRE(n1 <= nfft1 && n2 <= nfft2, "nfft must be >= size(s)");                             // :477
    DSP_REQUIRE(nfft1 < (int64_t(1) << 31) && nfft2 < (int64_t(1) << 31), "nfft too large");
    DSP_REQUIRE(ptype >= 0 && ptype <= 2 && r != 0.0, "bad ptype or r");
    return dtype == DSPB200_F64 ? periodogram2_run<double>(s, n1, n2, nfft1, nfft2, r, ptype, out, dev, st)
                                : periodogram2_run<float>(s, n1, n2, nfft1, nfft2, r, ptype, out, dev, st);
}
int dspb200_periodogram2_exec(int dtype, const void* s, int64_t n1, int64_t n2, int64_t nfft1, int64_t nfft2, double r, int ptype,
                              void* out) {
    DSP_RANGE("dspb200_periodogram2_exec");
    return periodogram2_entry(dtype, s, n1, n2, nfft1, nfft2, r, ptype, out, false, 0);
}
int dspb200_periodogram2_exec_dev(int dtype, const void* d_s, int64_t n1, int64_t n2, int64_t nfft1, int64_t nfft2, double r,
                                  int ptype, void* d_out, void* stream) {
    DSP_RANGE("dspb200_periodogram2_exec_dev");
    return periodogram2_entry(dtype, d_s, n1, n2, nfft1, nfft2, r, ptype, d_out, true, (cudaStream_t)stream);
}

int dspb200_spec_plan_destroy(dspb200_spec_plan* plan) {
    if (!plan) return DSPB200_OK;
    SpecPlanImpl* p = &plan->impl;
    if (p->d_window) cudaFree(p->d_window);
    if (p->d_tw) cudaFree(p->d_tw);
    if (p->d_t16) cudaFree(p->d_t16);
    if (p->d_t32) cudaFree(p->d_t32);
    if (p->d_t256) cudaFree(p->d_t256);
    p->partial.release(); p->segbuf.release(); p->specbuf.release(); p->acc.release();
    p->in[0].release(); p->in[1].release(); p->out.release(); p->tmp.release();
    if (p->fft_ok) cufftDestroy(p->fft);
    for (int i = 0; i < 2; ++i) {
        if (p->ev_in[i]) cudaEventDestroy(p->ev_in[i]);
        if (p->ev_done[i]) cudaEventDestroy(p->ev_done[i]);
    }
    if (p->s_copy) cudaStreamDestroy(p->s_copy);
    if (p->s_exec) cudaStreamDestroy(p->s_exec);
    delete plan;
    return DSPB200_OK;
}

}  // extern "C"
