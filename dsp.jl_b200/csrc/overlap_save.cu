// dspb200 -- overlap-save FFT convolution / filtering, single-FFT convolution, direct convolution.
//
// Reference path: unsafe_conv_kern_os! (src/dspbase.jl:490-609), os_prepare_conv / os_filter_transform! /
// os_conv_block! (:299-356), _fftfilt! (src/Filters/filt.jl:479-521), _conv_kern_fft! (src/dspbase.jl:611-644),
// _conv_td! (:646-660).
//
// Fused kernel (power-of-two nfft in shared memory): one CTA per block of L = nfft - nv + 1 outputs
//   global load (nv-1 sample halo, zero outside the signal) -> forward passes -> [last pass, x H, first pass of the
//   second transform in registers] -> remaining passes -> store the valid L samples.
// Each sample is read once and written once from/to HBM; the nv-1 halo re-read comes from L2.  Real signals ride two blocks per complex FFT (z = a + i b; h real => y = a*h + i b*h).
// H carries the 1/nfft of the unnormalised inverse (src/dspbase.jl:516, src/Filters/filt.jl:498).
#include "fft_core.cuh"
#include "fft_r32.cuh"
#include "async_copy.cuh"
#include <cufft.h>
#include <math.h>
#include <new>
#include <vector>

namespace dspb200 {

struct OsPlanImpl {
    int dtype = 0;
    bool cplx = false, f64 = false;
    int64_t nv = 0, nfft = 0, L = 0;
    bool fused = false;
    int device = 0;
    void* d_tw = nullptr;   // fused: last-pass twiddle table (fft_fill_tl)
    void* d_t16 = nullptr;  // fused: radix-16 twiddle tables
    void* d_t256 = nullptr;
    int sm_count = 148;
    int fused_per_sm = 0;   // resident CTAs per SM of this plan's fused kernel (occupancy calculator, asked once)
    void* d_t32 = nullptr;  // 16384-point Float32 plans: tables of the 32 x 32 x 16 kernel (fft_r32.cuh)
    void* d_t1024 = nullptr;
    void* d_H = nullptr;    // natural order; fused: cx<T>[nfft] pre-scaled by 1/nfft; generic: nfft or nfft/2+1 bins
    // generic
    cufftHandle fwd = 0, inv = 0;
    bool fft_ok = false;
    int64_t batch = 0, nbins = 0;
    DevBuf td, fd;
    // host path
    DevBuf in[2], out[2];
    cudaStream_t s_in = nullptr, s_exec = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_exec[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
};

template <typename T, bool CPLX> struct os_elt { using type = T; };
template <typename T> struct os_elt<T, true> { using type = cx<T>; };

// ---------------------------------------------------------------------------------------------- fused kernel
// Geometry (0-based): block q of a column produces outputs m in [out_begin + q*L, out_begin + (q+1)*L);
// its buffer slot j holds input sample i = out_begin + q*L - (nv-1) + j, and slot j >= nv-1 of the result
// is output m = out_begin + q*L + j - (nv-1).  Input samples outside [u_begin, u_begin+nu_local) are zero.
// Persistent CTAs stride over the units (unit = one complex block or two real blocks), neighbouring CTAs work
// on neighbouring blocks at the same time so the nv-1 sample halo is an L2 hit.
//
// One unit (fft_core.cuh):  first pass (global loads, thread c reads u[i0 + c + r N/16]: coalesced)  | middle passes |
// [last forward pass -> x H -> swap -> first pass of the second transform] in registers | middle passes | last pass ->
// global stores (thread t writes y[t + r N/16]: coalesced).  H is in natural order (the forward transform ends in
// natural order), pre-scaled by 1/N; thread t reads H[t + r N/16]: coalesced, no tiling needed.

// Launch shape of the fused kernel, tuned per size on the B200 (profiles/README.md, "resident threads" sweep):
//  * N = 512 .. 4096 (and the real N = 256 kernel): 1024 resident threads per SM under a 64-register cap, one radix-16
//    butterfly in flight per thread -- the extra warps hide the shared-memory latency (7-16 % faster than 512 threads
//    with two butterflies in flight under a 128-register cap);
//  * N = 8192: 512 resident threads, 128 registers, two butterflies in flight (the 64-register build spills there and
//    is 2-8 % slower).  Double precision: one CTA of up to 256 registers per thread.
// Float32 N = 16384 runs os_fused32_kernel instead.
template <typename T, int N, bool CPLX> struct os_threads {
    static constexpr bool f32 = sizeof(T) == 4;
    static constexpr int value = fft_threads<N>::value;
    static constexpr bool wide = f32 && ((N >= 512 && N <= 4096) || (N == 256 && !CPLX));     // 1024 resident threads
    static constexpr int minblocks = wide ? 1024 / value : fft_minblocks<T, N>::value;
};

template <typename T> __device__ __forceinline__ cx<T> ldg_cx(const cx<T>* __restrict__ p) {
    if constexpr (sizeof(T) == 4) {
        const float2 v = __ldg(reinterpret_cast<const float2*>(p));
        return mkc<T>(v.x, v.y);
    } else {
        const double2 v = __ldg(reinterpret_cast<const double2*>(p));
        return mkc<T>(v.x, v.y);
    }
}

// Per-unit geometry in slot coordinates j (0 <= j < N, block B of a real pair: j + L), 32-bit: u[j] is the sample in
// slot j, out[j] the output produced by slot j >= nv-1; slot j holds a stored sample iff jlo <= j < jhi, its output is
// wanted iff j < jend and is an exact zero (src/dspbase.jl:733-735) from jzero on.
template <typename E> struct OsUnit {
    const E* u;
    E* out;
    int jlo, jhi, jend, jzero;
    int nvm1, L;
};
__device__ __forceinline__ int os_clamp(int64_t v) {
    return (int)(v < -(int64_t(1) << 30) ? -(int64_t(1) << 30) : (v > (int64_t(1) << 30) ? (int64_t(1) << 30) : v));
}
// clamp(a - b) for a that may be INT64_MAX ("no limit") and |b| < 2^62: no signed overflow
__device__ __forceinline__ int os_clamp_diff(int64_t a, int64_t b) {
    return a >= (int64_t(1) << 62) ? (1 << 30) : os_clamp(a - b);
}

// Sample in slot j of a unit (block A in .x, block B of a real pair in .y).
// INTERIOR: every input sample of the unit is stored and every output is wanted and non-zero -- no bounds tests at all
// (all units but the first and the last few of a column)
template <typename T, bool CPLX, bool INTERIOR>
__device__ __forceinline__ cx<T> os_sample(const OsUnit<typename os_elt<T, CPLX>::type>& g, int j) {
    if constexpr (CPLX) {
        if constexpr (INTERIOR) return g.u[j];
        return (j >= g.jlo && j < g.jhi) ? g.u[j] : mkc<T>(T(0), T(0));
    } else {
        const int jb = j + g.L;
        if constexpr (INTERIOR) return mkc<T>(g.u[j], g.u[jb]);
        const T a = (j >= g.jlo && j < g.jhi) ? g.u[j] : T(0);
        const T b = (jb >= g.jlo && jb < g.jhi) ? g.u[jb] : T(0);
        return mkc<T>(a, b);
    }
}

// Output of slot j of a unit (y: swapped domain, result = (y.y, y.x)); slots below nv-1 produce none.
template <typename T, bool CPLX, bool INTERIOR>
__device__ __forceinline__ void os_put(const OsUnit<typename os_elt<T, CPLX>::type>& g, int j, cx<T> y) {
    if (j < g.nvm1) return;
    if constexpr (CPLX) {
        if constexpr (INTERIOR) g.out[j] = mkc<T>(y.y, y.x);
        else if (j < g.jend) g.out[j] = (j < g.jzero) ? mkc<T>(y.y, y.x) : mkc<T>(T(0), T(0));
    } else {
        const int jb = j + g.L;
        if constexpr (INTERIOR) {
            g.out[j] = y.y;
            g.out[jb] = y.x;
        } else {
            if (j < g.jend) g.out[j] = (j < g.jzero) ? y.y : T(0);
            if (jb < g.jend) g.out[jb] = (jb < g.jzero) ? y.x : T(0);
        }
    }
}

// One unit.  The samples are loaded inside the first pass.
template <typename T, int N, bool CPLX, int NT, bool INTERIOR>
__device__ __forceinline__ void os_unit(const FftCtx<T>& ctx, int tid, const OsUnit<typename os_elt<T, CPLX>::type>& g,
                                        const cx<T>* __restrict__ H) {
    constexpr int Q = fft_plan_traits<N>::Q;
    constexpr int ITERS = (Q + NT - 1) / NT;
    // the barrier inside (between the first butterfly and its stores) also ends the previous unit's last pass
    auto ld0 = [&](int j, int, int) -> cx<T> { return os_sample<T, CPLX, INTERIOR>(g, j); };
    fft_first_pass<T, N, NT, true>(ctx, tid, ld0);
    __syncthreads();
    fft_middle<T, N, NT>(ctx, tid);
    // last forward pass, x H, swap, first pass of the second transform -- in registers
    cx<T> v[ITERS][16];
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int tp = tid + it * NT;
        if (Q % NT == 0 || tp < Q) {
            fft_last_pass<T, N, (ITERS == 1 && Q % NT == 0) ? NT : 0>(ctx, tp, v[it], tid);
#pragma unroll
            for (int r = 0; r < 16; ++r) v[it][r] = cswap(cmul(v[it][r], ldg_cx<T>(H + tp + r * Q)));
            fft_bfly16_plain<T>(v[it]);
        }
    }
    __syncthreads();                                   // every thread has read its last-pass inputs
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int tp = tid + it * NT;
        if (Q % NT == 0 || tp < Q) fft_store_block<T, N>(ctx.sm, tp, v[it]);
    }
    __syncthreads();
    fft_middle<T, N, NT>(ctx, tid);
    // Last pass, streamed one radix-RL butterfly at a time: RL live values instead of 16
    constexpr int RL = fft_plan_traits<N>::RL, NBF = 16 / RL;
    auto chunk = [&](auto a_, int tp) {
        constexpr int A = decltype(a_)::value;
        cx<T> u[RL];
        fft_last_pass_chunk<T, N, A>(ctx, tp, u);
#pragma unroll
        for (int jj = 0; jj < RL; ++jj) os_put<T, CPLX, INTERIOR>(g, tp + (A + NBF * jj) * Q, u[jj]);
    };
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int tp = tid + it * NT;
        if (Q % NT != 0 && tp >= Q) break;
        chunk(std::integral_constant<int, 0>{}, tp);
        if constexpr (NBF >= 2) chunk(std::integral_constant<int, 1>{}, tp);
        if constexpr (NBF >= 4) { chunk(std::integral_constant<int, 2>{}, tp); chunk(std::integral_constant<int, 3>{}, tp); }
        if constexpr (NBF >= 8) {
            chunk(std::integral_constant<int, 4>{}, tp); chunk(std::integral_constant<int, 5>{}, tp);
            chunk(std::integral_constant<int, 6>{}, tp); chunk(std::integral_constant<int, 7>{}, tp);
        }
    }
}

template <typename T, int N, bool CPLX>
__global__ void __launch_bounds__((os_threads<T, N, CPLX>::value), (os_threads<T, N, CPLX>::minblocks))
os_fused_kernel(const void* __restrict__ u_, int64_t u_begin, int64_t nu_local, int64_t u_col_stride,
                void* __restrict__ out_, int64_t out_begin, int64_t out_count, int64_t out_col_stride,
                int64_t zero_from, int nv, int64_t units_per_col, int64_t total_units, const cx<T>* __restrict__ gtl,
                const cx<T>* __restrict__ g16, const cx<T>* __restrict__ g256, const cx<T>* __restrict__ H) {
    constexpr int NT = os_threads<T, N, CPLX>::value;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* sm = reinterpret_cast<cx<T>*>(smem_raw);
    using E = typename os_elt<T, CPLX>::type;
    const int tid = threadIdx.x;
    pdl_launch_dependents();
    const FftCtx<T> ctx = fft_make_ctx<T, N, NT>(sm, g16, g256, gtl, tid);
    pdl_wait();                                        // tables staged; from here on data of preceding kernels is touched
    __syncthreads();
    const int L = N - nv + 1;
    const int span = CPLX ? N : N + L;                 // input samples / output range (+ nv - 1) of one unit
    const bool onecol = units_per_col >= total_units;
    // geometry of unit gu; returns whether it is interior
    auto geometry = [&](int64_t gu, OsUnit<E>& g) -> bool {
        const int64_t col = onecol ? 0 : gu / units_per_col;
        const int64_t unit = gu - col * units_per_col;
        const int64_t q = CPLX ? unit : 2 * unit;
        const int64_t s0 = out_begin + q * L - (nv - 1);          // global index of the sample in slot 0
        const int64_t i0 = s0 - u_begin;                          // its local index
        g.u = reinterpret_cast<const E*>(u_) + col * u_col_stride + i0;
        g.out = reinterpret_cast<E*>(out_) + col * out_col_stride + (s0 - out_begin);
        g.jlo = os_clamp(-i0);
        g.jhi = os_clamp(nu_local - i0);
        g.jend = os_clamp(out_begin + out_count - s0);
        g.jzero = os_clamp_diff(zero_from, s0);
        g.nvm1 = nv - 1;
        g.L = L;
        return g.jlo <= 0 && g.jhi >= span && g.jend >= span && g.jzero >= span;
    };
    // pull the input range of unit gn into L2 (16-byte aligned sub-range, clipped to the stored signal)
    auto l2_prefetch = [&](int64_t gn) {
        if (tid == 0 && gn < total_units) {
            const int64_t coln = onecol ? 0 : gn / units_per_col;
            const int64_t qn = (CPLX ? 1 : 2) * (gn - coln * units_per_col);
            int64_t lo = out_begin + qn * L - (nv - 1) - u_begin;
            int64_t hi = lo + span;
            if (lo < 0) lo = 0;
            if (hi > nu_local) hi = nu_local;
            const uintptr_t a0 = ((uintptr_t)(reinterpret_cast<const E*>(u_) + coln * u_col_stride + lo) + 15) & ~(uintptr_t)15;
            const uintptr_t a1 = (uintptr_t)(reinterpret_cast<const E*>(u_) + coln * u_col_stride + hi) & ~(uintptr_t)15;
            if (hi > lo && a1 > a0) tma_prefetch_l2(reinterpret_cast<const void*>(a0), (uint32_t)(a1 - a0));
        }
    };
    for (int64_t gu = blockIdx.x; gu < total_units; gu += gridDim.x) {
        l2_prefetch(gu + (int64_t)gridDim.x);          // this CTA's next unit, pulled into L2 while this one computes
        OsUnit<E> g;
        if (geometry(gu, g)) os_unit<T, N, CPLX, NT, true>(ctx, tid, g, H);
        else os_unit<T, N, CPLX, NT, false>(ctx, tid, g, H);
    }
}

// ---------------------------------------------------------------------------------------------- 32 x 32 x 16 kernel
// The 16384-point Float32 block as 32 x 32 x 16 (fft_r32.cuh): 512 threads, one radix-32 butterfly per thread in the first
// and the middle pass, two radix-16 butterflies in the last one.  Same unit geometry, same H, same results up to rounding.
// It runs every 16384-point Float32 plan (2^26 ComplexF32 samples, 4097 taps: 0.489 ms against 0.520 ms for 16 x 16 x 16 x 4;
// real Float32: 0.269 against 0.274 ms; measured in round 2 with a variant since removed; see the history before this commit).
template <typename T, bool CPLX, bool INTERIOR>
__device__ __forceinline__ void os_unit32(const r32::Ctx<T>& ctx, int tid, const OsUnit<typename os_elt<T, CPLX>::type>& g,
                                          const cx<T>* __restrict__ H) {
    cx<T> v[32];
#pragma unroll
    for (int r = 0; r < 32; ++r) v[r] = os_sample<T, CPLX, INTERIOR>(g, tid + r * r32::Q32);
    fft_bfly<T, 32, true>(v, nullptr);
    __syncthreads();                                   // the previous unit's last pass has read the buffer
    r32::store_block<T>(ctx.sm, tid, v);
    __syncthreads();
    r32::middle_pass<T>(ctx, tid);
    __syncthreads();
    {
        // last forward pass of the butterflies tid and tid + 512, x H, swap: together they hold Y[tid + 512 m], m < 32,
        // the inputs of the plain first-pass butterfly of residue class tid of the second transform.  H is requested
        // after both butterflies' shared-memory loads.
        cx<T> a[16], b[16];
        r32::last_pass<T>(ctx, tid, a);
        r32::last_pass<T>(ctx, tid + r32::Q32, b);
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            v[2 * r] = cswap(cmul(a[r], ldg_cx<T>(H + tid + r * r32::Q16)));
            v[2 * r + 1] = cswap(cmul(b[r], ldg_cx<T>(H + tid + r32::Q32 + r * r32::Q16)));
        }
    }
    fft_bfly<T, 32, true>(v, nullptr);
    __syncthreads();                                   // every thread has read its last-pass inputs
    r32::store_block<T>(ctx.sm, tid, v);
    __syncthreads();
    r32::middle_pass<T>(ctx, tid);
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        const int tp = tid + it * r32::Q32;
        cx<T> y[16];
        r32::last_pass<T>(ctx, tp, y);
#pragma unroll
        for (int r = 0; r < 16; ++r) os_put<T, CPLX, INTERIOR>(g, tp + r * r32::Q16, y[r]);
    }
}

template <typename T, bool CPLX>
__global__ void __launch_bounds__(r32::NT, 1)
os_fused32_kernel(const void* __restrict__ u_, int64_t u_begin, int64_t nu_local, int64_t u_col_stride,
                  void* __restrict__ out_, int64_t out_begin, int64_t out_count, int64_t out_col_stride,
                  int64_t zero_from, int nv, int64_t units_per_col, int64_t total_units, const cx<T>* __restrict__ g32,
                  const cx<T>* __restrict__ g1024, const cx<T>* __restrict__ H) {
    constexpr int N = r32::N;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    using E = typename os_elt<T, CPLX>::type;
    const int tid = threadIdx.x;
    pdl_launch_dependents();
    const r32::Ctx<T> ctx = r32::make_ctx<T>(reinterpret_cast<cx<T>*>(smem_raw), g32, g1024, tid);
    pdl_wait();                                        // tables staged; from here on data of preceding kernels is touched
    __syncthreads();
    // Unit geometry and L2 prefetch as in os_fused_kernel, written out: shared with it as helpers, they changed this
    // kernel's SASS and cost 0.15 % of the bench conv stage (B200, 1000 W power limit).
    const int L = N - nv + 1;
    const int span = CPLX ? N : N + L;
    const bool onecol = units_per_col >= total_units;
    for (int64_t gu = blockIdx.x; gu < total_units; gu += gridDim.x) {
        const int64_t col = onecol ? 0 : gu / units_per_col;
        const int64_t unit = gu - col * units_per_col;
        const int64_t q = CPLX ? unit : 2 * unit;
        const int64_t s0 = out_begin + q * L - (nv - 1);
        const int64_t i0 = s0 - u_begin;
        OsUnit<E> g;
        g.u = reinterpret_cast<const E*>(u_) + col * u_col_stride + i0;
        g.out = reinterpret_cast<E*>(out_) + col * out_col_stride + (s0 - out_begin);
        g.jlo = os_clamp(-i0);
        g.jhi = os_clamp(nu_local - i0);
        g.jend = os_clamp(out_begin + out_count - s0);
        g.jzero = os_clamp_diff(zero_from, s0);
        g.nvm1 = nv - 1;
        g.L = L;
        const bool interior = g.jlo <= 0 && g.jhi >= span && g.jend >= span && g.jzero >= span;
        // pull the input range of this CTA's next unit into L2 while this one computes
        if (tid == 0 && gu + gridDim.x < total_units) {
            const int64_t gn = gu + gridDim.x;
            const int64_t coln = onecol ? 0 : gn / units_per_col;
            const int64_t qn = (CPLX ? 1 : 2) * (gn - coln * units_per_col);
            int64_t lo = out_begin + qn * L - (nv - 1) - u_begin;
            int64_t hi = lo + span;
            if (lo < 0) lo = 0;
            if (hi > nu_local) hi = nu_local;
            const uintptr_t a0 = ((uintptr_t)(reinterpret_cast<const E*>(u_) + coln * u_col_stride + lo) + 15) & ~(uintptr_t)15;
            const uintptr_t a1 = (uintptr_t)(reinterpret_cast<const E*>(u_) + coln * u_col_stride + hi) & ~(uintptr_t)15;
            if (hi > lo && a1 > a0) tma_prefetch_l2(reinterpret_cast<const void*>(a0), (uint32_t)(a1 - a0));
        }
        if (interior) os_unit32<T, CPLX, true>(ctx, tid, g, H);
        else os_unit32<T, CPLX, false>(ctx, tid, g, H);
    }
}

// H in natural order: forward transform of the zero-padded taps, scaled by 1/N.
template <typename T, int N, bool CPLX>
__global__ void __launch_bounds__(fft_threads<N>::value, fft_minblocks<T, N>::value)
os_filter_kernel(const void* __restrict__ v_, int nv, const cx<T>* __restrict__ gtl, const cx<T>* __restrict__ g16,
                 const cx<T>* __restrict__ g256, cx<T>* __restrict__ H) {
    constexpr int NT = fft_threads<N>::value;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    cx<T>* sm = reinterpret_cast<cx<T>*>(smem_raw);
    using E = typename os_elt<T, CPLX>::type;
    const E* v = reinterpret_cast<const E*>(v_);
    const FftCtx<T> ctx = fft_make_ctx<T, N, NT>(sm, g16, g256, gtl, threadIdx.x);
    __syncthreads();
    const T scale = T(1) / T(N);
    auto ld0 = [&](int j, int, int) -> cx<T> {
        if (j >= nv) return mkc<T>(T(0), T(0));
        if constexpr (CPLX) return v[j]; else return mkc<T>(v[j], T(0));
    };
    auto stl = [&](int k, int, int, cx<T> x) { H[k] = cscale(x, scale); };
    fft_forward<T, N, NT>(ctx, threadIdx.x, ld0, stl);
}

// ---------------------------------------------------------------------------------------------- generic kernels
template <typename T, bool CPLX>
__global__ void os_gather_kernel(const void* __restrict__ u_, int64_t u_begin, int64_t nu_local, int64_t m_first,
                                 int64_t L, int64_t nv, int64_t nfft, int64_t nblk, void* __restrict__ td_) {
    using E = typename os_elt<T, CPLX>::type;
    const E* u = reinterpret_cast<const E*>(u_);
    E* td = reinterpret_cast<E*>(td_);
    const int64_t total = nblk * nfft;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / nfft, j = i - b * nfft;
        const int64_t src = m_first + b * L - (nv - 1) + j - u_begin;
        E v;
        if constexpr (CPLX) v = mkc<T>(T(0), T(0)); else v = T(0);
        if (src >= 0 && src < nu_local) v = u[src];
        td[i] = v;
    }
}

template <typename T>
__global__ void os_cmul_kernel(cx<T>* __restrict__ X, const cx<T>* __restrict__ H, int64_t nbins, int64_t nblk) {
    const int64_t total = nblk * nbins;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
        X[i] = cmul(X[i], H[i % nbins]);
}

// ---------------------------------------------------------------------------------------------- hilbert
// hilbert(x), src/util.jl:31-75: X = rfft(x) written into the first n/2+1 bins of a zeroed length-n complex buffer,
// bins 2 .. n/2 + isodd(n) (1-based) doubled, inverse complex FFT with the 1/n normalisation.
template <typename T>
__global__ void hilbert_weight_kernel(cx<T>* __restrict__ X, int64_t n, int64_t ncols, T scale) {
    const int64_t total = n * ncols;
    const int64_t last2 = (n + 1) / 2 - 1;                    // last doubled bin (0-based)
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = i % n;
        if (k > n / 2) { X[i] = mkc<T>(T(0), T(0)); continue; }      // never written by the real transform
        const T w = (k >= 1 && k <= last2) ? T(2) * scale : scale;   // DC and (n even) Nyquist keep weight 1
        X[i] = cscale(X[i], w);
    }
}

// ---------------------------------------------------------------------------------------------- N-D conv (rank <= 3)
// Column-major arrays, dim 1 fastest (Julia layout); ranks below 3 carry trailing sizes of 1.
struct Dims3 { int64_t n[3]; };

// dst (size d) = src (size s) zero-padded / cropped at the origin: _zeropad!, src/dspbase.jl:187-256, and the copyto! of
// the valid region, :624-627 / :640-643
template <typename E>
__global__ void nd_copy_kernel(const E* __restrict__ src, Dims3 s, E* __restrict__ dst, Dims3 d, E zero) {
    const int64_t total = d.n[0] * d.n[1] * d.n[2];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i0 = i % d.n[0], i1 = (i / d.n[0]) % d.n[1], i2 = i / (d.n[0] * d.n[1]);
        dst[i] = (i0 < s.n[0] && i1 < s.n[1] && i2 < s.n[2]) ? src[i0 + s.n[0] * (i1 + s.n[1] * i2)] : zero;
    }
}

// _conv_td!, src/dspbase.jl:646-660, N-D: out[k] = sum over m of u[m] * v[k - m] (muladd), one output per thread
template <typename T, bool CPLX>
__global__ void conv_direct_nd_kernel(const void* __restrict__ u_, Dims3 su, const void* __restrict__ v_, Dims3 sv,
                                      void* __restrict__ out_) {
    using E = typename os_elt<T, CPLX>::type;
    const E* u = reinterpret_cast<const E*>(u_);
    const E* v = reinterpret_cast<const E*>(v_);
    E* out = reinterpret_cast<E*>(out_);
    const int64_t o0 = su.n[0] + sv.n[0] - 1, o1 = su.n[1] + sv.n[1] - 1, o2 = su.n[2] + sv.n[2] - 1;
    const int64_t total = o0 * o1 * o2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k0 = i % o0, k1 = (i / o0) % o1, k2 = i / (o0 * o1);
        T ar = T(0), ai = T(0);
        for (int64_t m2 = max(k2 - (sv.n[2] - 1), (int64_t)0); m2 <= min(k2, su.n[2] - 1); ++m2)
            for (int64_t m1 = max(k1 - (sv.n[1] - 1), (int64_t)0); m1 <= min(k1, su.n[1] - 1); ++m1)
                for (int64_t m0 = max(k0 - (sv.n[0] - 1), (int64_t)0); m0 <= min(k0, su.n[0] - 1); ++m0) {
                    const E a = u[m0 + su.n[0] * (m1 + su.n[1] * m2)];
                    const E b = v[(k0 - m0) + sv.n[0] * ((k1 - m1) + sv.n[1] * (k2 - m2))];
                    if constexpr (CPLX) {
                        ar = fma(a.x, b.x, fma(-a.y, b.y, ar));
                        ai = fma(a.x, b.y, fma(a.y, b.x, ai));
                    } else {
                        ar = fma(a, b, ar);
                    }
                }
        if constexpr (CPLX) out[i] = mkc<T>(ar, ai); else out[i] = ar;
    }
}

// N-D overlap-save blocking: unsafe_conv_kern_os! with its perimeter blocks, src/dspbase.jl:371-609.  Block b = (b0, b1, b2)
// of the nb grid owns the outputs L .* b .. L .* (b + 1) - 1 (L = save_blocksize, :505); its time-domain buffer holds nf
// samples per dimension starting sv - 1 before the block's first output and is zero where that lies outside u (the
// reference's pad_before / pad_after, :449-463; centre blocks, :583-606, are the case without padding).  Blocks are
// transformed `nblk` at a time by ONE batched N-D cuFFT plan; blocks past the end of the grid (last batch) are zeros.
struct OsNd { int64_t su[3], sv[3], so[3], nf[3], L[3], nb[3]; };

template <typename E>
__global__ void nd_os_gather_kernel(const E* __restrict__ u, OsNd g, int64_t blk0, int64_t nblk, E* __restrict__ td, E zero) {
    const int64_t per = g.nf[0] * g.nf[1] * g.nf[2], total = per * nblk, nblocks = g.nb[0] * g.nb[1] * g.nb[2];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = blk0 + i / per, r = i % per;
        E val = zero;
        if (b < nblocks) {
            const int64_t i0 = r % g.nf[0], i1 = (r / g.nf[0]) % g.nf[1], i2 = r / (g.nf[0] * g.nf[1]);
            const int64_t b0 = b % g.nb[0], b1 = (b / g.nb[0]) % g.nb[1], b2 = b / (g.nb[0] * g.nb[1]);
            const int64_t s0 = g.L[0] * b0 - (g.sv[0] - 1) + i0, s1 = g.L[1] * b1 - (g.sv[1] - 1) + i1,
                          s2 = g.L[2] * b2 - (g.sv[2] - 1) + i2;
            if (s0 >= 0 && s0 < g.su[0] && s1 >= 0 && s1 < g.su[1] && s2 >= 0 && s2 < g.su[2])
                val = u[s0 + g.su[0] * (s1 + g.su[1] * s2)];
        }
        td[i] = val;
    }
}

// the valid region sv : nf of every block (:603-606, cropped at the end of the output, :468-482) -> out
template <typename E>
__global__ void nd_os_scatter_kernel(const E* __restrict__ td, OsNd g, int64_t blk0, int64_t nblk, E* __restrict__ out) {
    const int64_t per = g.L[0] * g.L[1] * g.L[2], total = per * nblk, nblocks = g.nb[0] * g.nb[1] * g.nb[2];
    const int64_t nfp = g.nf[0] * g.nf[1] * g.nf[2];
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t lb = i / per, b = blk0 + lb, r = i % per;
        if (b >= nblocks) continue;
        const int64_t j0 = r % g.L[0], j1 = (r / g.L[0]) % g.L[1], j2 = r / (g.L[0] * g.L[1]);
        const int64_t b0 = b % g.nb[0], b1 = (b / g.nb[0]) % g.nb[1], b2 = b / (g.nb[0] * g.nb[1]);
        const int64_t o0 = g.L[0] * b0 + j0, o1 = g.L[1] * b1 + j1, o2 = g.L[2] * b2 + j2;
        if (o0 < g.so[0] && o1 < g.so[1] && o2 < g.so[2])
            out[o0 + g.so[0] * (o1 + g.so[1] * o2)] =
                td[lb * nfp + (j0 + g.sv[0] - 1) + g.nf[0] * ((j1 + g.sv[1] - 1) + g.nf[1] * (j2 + g.sv[2] - 1))];
    }
}

template <typename T, bool CPLX>
__global__ void os_scatter_kernel(const void* __restrict__ td_, int64_t m_first, int64_t L, int64_t nv, int64_t nfft,
                                  int64_t nblk, void* __restrict__ out_, int64_t out_begin, int64_t out_end,
                                  int64_t zero_from) {
    using E = typename os_elt<T, CPLX>::type;
    const E* td = reinterpret_cast<const E*>(td_);
    E* out = reinterpret_cast<E*>(out_);
    const int64_t total = nblk * L;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / L, j = i - b * L;
        const int64_t m = m_first + b * L + j;
        if (m < out_end) {
            E v = td[b * nfft + (nv - 1) + j];
            if (m >= zero_from) { if constexpr (CPLX) v = mkc<T>(T(0), T(0)); else v = T(0); }
            out[m - out_begin] = v;
        }
    }
}

template <typename T, bool CPLX>
__global__ void pad_copy_kernel(const void* __restrict__ src_, int64_t n, void* __restrict__ dst_, int64_t nfft, T scale) {
    using E = typename os_elt<T, CPLX>::type;
    const E* src = reinterpret_cast<const E*>(src_);
    E* dst = reinterpret_cast<E*>(dst_);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nfft; i += (int64_t)gridDim.x * blockDim.x) {
        E v;
        if constexpr (CPLX) v = mkc<T>(T(0), T(0)); else v = T(0);
        if (i < n) {
            v = src[i];
            if constexpr (CPLX) v = cscale(v, scale); else v = v * scale;
        }
        dst[i] = v;
    }
}

template <typename T>
__global__ void scale_cplx_kernel(cx<T>* __restrict__ X, int64_t n, T scale) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        X[i] = cscale(X[i], scale);
}

// direct convolution, src/dspbase.jl:646-660: out[k] = sum_n large[n] * small[k-n], n ascending, muladd
template <typename T, bool CPLX>
__global__ void conv_direct_kernel(const void* __restrict__ large_, int64_t nl, const void* __restrict__ small_,
                                   int64_t ns, void* __restrict__ out_) {
    using E = typename os_elt<T, CPLX>::type;
    const E* large = reinterpret_cast<const E*>(large_);
    const E* small = reinterpret_cast<const E*>(small_);
    E* out = reinterpret_cast<E*>(out_);
    const int64_t nout = nl + ns - 1;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < nout; k += (int64_t)gridDim.x * blockDim.x) {
        const int64_t lo = k - (ns - 1) > 0 ? k - (ns - 1) : 0;
        const int64_t hi = k < nl - 1 ? k : nl - 1;
        if constexpr (CPLX) {
            cx<T> acc = mkc<T>(T(0), T(0));
            for (int64_t n = lo; n <= hi; ++n) {
                const cx<T> a = large[n], b = small[k - n];
                acc.x = fma(a.x, b.x, fma(-a.y, b.y, acc.x));
                acc.y = fma(a.x, b.y, fma(a.y, b.x, acc.y));
            }
            out[k] = acc;
        } else {
            T acc = T(0);
            for (int64_t n = lo; n <= hi; ++n) acc = fma(large[n], small[k - n], acc);
            out[k] = acc;
        }
    }
}

// ---------------------------------------------------------------------------------------------- dispatch
#define DSP_OS_SIZES(X) X(32) X(64) X(128) X(256) X(512) X(1024) X(2048) X(4096) X(8192) X(16384)

static bool os_fused_ok(int64_t nfft, int64_t nv, bool f64) {
    if (nfft < 32 || (nfft & (nfft - 1))) return false;
    if (nfft > (f64 ? 8192 : 16384)) return false;
    return nfft >= nv;
}

template <typename K> static int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) DSP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return DSPB200_OK;
}

struct OsRange {
    const void* u; int64_t u_begin, nu_local, u_col_stride;
    void* out; int64_t out_begin, out_count, out_col_stride;
    int64_t zero_from, ncols;
};

template <typename T, int N, bool CPLX>
static int launch_os_fused(OsPlanImpl* p, const OsRange& a, cudaStream_t st) {
    constexpr int NT = os_threads<T, N, CPLX>::value;
    const size_t smem = (size_t)fft_smem_elems<T, N>() * sizeof(cx<T>);
    auto kern = os_fused_kernel<T, N, CPLX>;
    const int64_t nblk = cdiv(a.out_count, p->L);
    const int64_t upc = CPLX ? nblk : (nblk + 1) / 2;
    const int64_t units = upc * a.ncols;
    if (units < 1) return DSPB200_OK;
    // persistent grid: one resident wave (CTAs per SM from the occupancy calculator: shared memory and register cap)
    if (p->fused_per_sm < 1) {
        DSP_TRY(set_smem(kern, smem));
        int per = 1;
        DSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kern, NT, smem));
        p->fused_per_sm = per < 1 ? 1 : per;
    }
    const int per_sm = p->fused_per_sm;
    const int64_t cap = (int64_t)p->sm_count * per_sm;
    const int64_t blocks = units < cap ? units : cap;
    DSP_CUDA(launch_pdl(kern, (unsigned)blocks, NT, smem, st, a.u, a.u_begin, a.nu_local, a.u_col_stride, a.out, a.out_begin,
                        a.out_count, a.out_col_stride, a.zero_from, (int)p->nv, upc, units,
                        reinterpret_cast<const cx<T>*>(p->d_tw), reinterpret_cast<const cx<T>*>(p->d_t16),
                        reinterpret_cast<const cx<T>*>(p->d_t256), reinterpret_cast<const cx<T>*>(p->d_H)));
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

template <bool CPLX>
static int launch_os_fused32(OsPlanImpl* p, const OsRange& a, cudaStream_t st) {
    const size_t smem = (size_t)r32::smem_elems<float>() * sizeof(cx<float>);
    auto kern = os_fused32_kernel<float, CPLX>;
    const int64_t nblk = cdiv(a.out_count, p->L);
    const int64_t upc = CPLX ? nblk : (nblk + 1) / 2;
    const int64_t units = upc * a.ncols;
    if (units < 1) return DSPB200_OK;
    DSP_TRY(set_smem(kern, smem));
    const int64_t cap = p->sm_count;                               // one CTA per SM (213 KB of shared memory)
    const int64_t blocks = units < cap ? units : cap;
    DSP_CUDA(launch_pdl(kern, (unsigned)blocks, r32::NT, smem, st, a.u, a.u_begin, a.nu_local, a.u_col_stride, a.out,
                        a.out_begin, a.out_count, a.out_col_stride, a.zero_from, (int)p->nv, upc, units,
                        reinterpret_cast<const cx<float>*>(p->d_t32), reinterpret_cast<const cx<float>*>(p->d_t1024),
                        reinterpret_cast<const cx<float>*>(p->d_H)));
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

template <typename T> static int os_fused_dispatch(OsPlanImpl* p, const OsRange& a, cudaStream_t st) {
    if constexpr (sizeof(T) == 4) {
        if (p->nfft == 16384) return p->cplx ? launch_os_fused32<true>(p, a, st) : launch_os_fused32<false>(p, a, st);
    }
    switch (p->nfft) {
#define X(NN)                                                                                   \
    case NN:                                                                                    \
        if constexpr (NN > 8192) break;      /* Float32: os_fused32_kernel above; Float64 is not fused */ \
        else return p->cplx ? launch_os_fused<T, NN, true>(p, a, st) : launch_os_fused<T, NN, false>(p, a, st);
        DSP_OS_SIZES(X)
#undef X
    }
    set_error("no fused overlap-save kernel for nfft=%lld", (long long)p->nfft);
    return DSPB200_EUNSUPPORTED;
}

template <typename T, int N, bool CPLX>
static int launch_os_filter(OsPlanImpl* p, const void* d_v) {
    constexpr int NT = fft_threads<N>::value;
    const size_t smem = (size_t)fft_smem_elems<T, N>() * sizeof(cx<T>);
    auto kern = os_filter_kernel<T, N, CPLX>;
    DSP_TRY(set_smem(kern, smem));
    kern<<<1, NT, smem, 0>>>(d_v, (int)p->nv, reinterpret_cast<const cx<T>*>(p->d_tw), reinterpret_cast<const cx<T>*>(p->d_t16),
                             reinterpret_cast<const cx<T>*>(p->d_t256), reinterpret_cast<cx<T>*>(p->d_H));
    DSP_LAUNCH_OK();
    DSP_CUDA(cudaStreamSynchronize(0));
    return DSPB200_OK;
}

template <typename T> static int os_filter_dispatch(OsPlanImpl* p, const void* d_v) {
    switch (p->nfft) {
#define X(NN)                                                                                   \
    case NN:                                                                                    \
        if constexpr (sizeof(T) == 8 && NN > 8192) break;                                       \
        else return p->cplx ? launch_os_filter<T, NN, true>(p, d_v) : launch_os_filter<T, NN, false>(p, d_v);
        DSP_OS_SIZES(X)
#undef X
    }
    return DSPB200_EUNSUPPORTED;
}

static int cufft_fail(cufftResult r, const char* what) {
    set_error("cuFFT error %d in %s", (int)r, what);
    return DSPB200_ECUFFT;
}
#define DSP_CUFFT(call)                                          \
    do {                                                         \
        cufftResult r__ = (call);                                \
        if (r__ != CUFFT_SUCCESS) return cufft_fail(r__, #call); \
    } while (0)

static int grid_for(int64_t total, int threads) {
    int64_t g = cdiv(total, threads);
    if (g > 148 * 64) g = 148 * 64;
    if (g < 1) g = 1;
    return (int)g;
}

// forward / inverse transforms of `batch` rows held in td (time) and fd (frequency)
static int generic_exec_fwd(OsPlanImpl* p, cufftHandle h, void* td, void* fd, cudaStream_t st) {
    DSP_CUFFT(cufftSetStream(h, st));
    if (p->cplx) {
        if (p->f64) DSP_CUFFT(cufftExecZ2Z(h, (cufftDoubleComplex*)td, (cufftDoubleComplex*)fd, CUFFT_FORWARD));
        else DSP_CUFFT(cufftExecC2C(h, (cufftComplex*)td, (cufftComplex*)fd, CUFFT_FORWARD));
    } else {
        if (p->f64) DSP_CUFFT(cufftExecD2Z(h, (cufftDoubleReal*)td, (cufftDoubleComplex*)fd));
        else DSP_CUFFT(cufftExecR2C(h, (cufftReal*)td, (cufftComplex*)fd));
    }
    count_launch(1);
    return DSPB200_OK;
}
static int generic_exec_inv(OsPlanImpl* p, cufftHandle h, void* fd, void* td, cudaStream_t st) {
    DSP_CUFFT(cufftSetStream(h, st));
    if (p->cplx) {
        if (p->f64) DSP_CUFFT(cufftExecZ2Z(h, (cufftDoubleComplex*)fd, (cufftDoubleComplex*)td, CUFFT_INVERSE));
        else DSP_CUFFT(cufftExecC2C(h, (cufftComplex*)fd, (cufftComplex*)td, CUFFT_INVERSE));
    } else {
        if (p->f64) DSP_CUFFT(cufftExecZ2D(h, (cufftDoubleComplex*)fd, (cufftDoubleReal*)td));
        else DSP_CUFFT(cufftExecC2R(h, (cufftComplex*)fd, (cufftReal*)td));
    }
    count_launch(1);
    return DSPB200_OK;
}

static int make_plans(bool cplx, bool f64, int64_t nfft, int64_t batch, cufftHandle* fwd, cufftHandle* inv) {
    long long nn[1] = {(long long)nfft};
    size_t ws = 0;
    DSP_CUFFT(cufftCreate(fwd));
    DSP_CUFFT(cufftCreate(inv));
    if (cplx) {
        const cufftType t = f64 ? CUFFT_Z2Z : CUFFT_C2C;
        DSP_CUFFT(cufftMakePlanMany64(*fwd, 1, nn, nullptr, 1, 0, nullptr, 1, 0, t, batch, &ws));
        DSP_CUFFT(cufftMakePlanMany64(*inv, 1, nn, nullptr, 1, 0, nullptr, 1, 0, t, batch, &ws));
    } else {
        DSP_CUFFT(cufftMakePlanMany64(*fwd, 1, nn, nullptr, 1, 0, nullptr, 1, 0, f64 ? CUFFT_D2Z : CUFFT_R2C, batch, &ws));
        DSP_CUFFT(cufftMakePlanMany64(*inv, 1, nn, nullptr, 1, 0, nullptr, 1, 0, f64 ? CUFFT_Z2D : CUFFT_C2R, batch, &ws));
    }
    return DSPB200_OK;
}

template <typename T> static int os_generic_run(OsPlanImpl* p, const OsRange& a, cudaStream_t st) {
    const int threads = 256;
    for (int64_t c = 0; c < a.ncols; ++c) {
        const char* ucol = (const char*)a.u + (size_t)(c * a.u_col_stride) * dtype_size(p->dtype);
        char* ocol = (char*)a.out + (size_t)(c * a.out_col_stride) * dtype_size(p->dtype);
        const int64_t nblk_total = cdiv(a.out_count, p->L);
        for (int64_t b0 = 0; b0 < nblk_total; b0 += p->batch) {
            const int64_t nblk = nblk_total - b0 < p->batch ? nblk_total - b0 : p->batch;
            const int64_t m_first = a.out_begin + b0 * p->L;
            // gather all `batch` rows (rows >= nblk read past the range and are simply ignored by scatter)
            if (p->cplx) os_gather_kernel<T, true><<<grid_for(p->batch * p->nfft, threads), threads, 0, st>>>(ucol, a.u_begin, a.nu_local, m_first, p->L, p->nv, p->nfft, p->batch, p->td.p);
            else os_gather_kernel<T, false><<<grid_for(p->batch * p->nfft, threads), threads, 0, st>>>(ucol, a.u_begin, a.nu_local, m_first, p->L, p->nv, p->nfft, p->batch, p->td.p);
            DSP_LAUNCH_OK();
            DSP_TRY(generic_exec_fwd(p, p->fwd, p->td.p, p->fd.p, st));
            os_cmul_kernel<T><<<grid_for(p->batch * p->nbins, threads), threads, 0, st>>>(reinterpret_cast<cx<T>*>(p->fd.p), reinterpret_cast<const cx<T>*>(p->d_H), p->nbins, p->batch);
            DSP_LAUNCH_OK();
            DSP_TRY(generic_exec_inv(p, p->inv, p->fd.p, p->td.p, st));
            if (p->cplx) os_scatter_kernel<T, true><<<grid_for(nblk * p->L, threads), threads, 0, st>>>(p->td.p, m_first, p->L, p->nv, p->nfft, nblk, ocol, a.out_begin, a.out_begin + a.out_count, a.zero_from);
            else os_scatter_kernel<T, false><<<grid_for(nblk * p->L, threads), threads, 0, st>>>(p->td.p, m_first, p->L, p->nv, p->nfft, nblk, ocol, a.out_begin, a.out_begin + a.out_count, a.zero_from);
            DSP_LAUNCH_OK();
        }
    }
    return DSPB200_OK;
}

static int os_run(OsPlanImpl* p, const OsRange& a, cudaStream_t st) {
    if (a.out_count <= 0 || a.ncols <= 0) return DSPB200_OK;
    if (p->fused) return p->f64 ? os_fused_dispatch<double>(p, a, st) : os_fused_dispatch<float>(p, a, st);
    return p->f64 ? os_generic_run<double>(p, a, st) : os_generic_run<float>(p, a, st);
}

static int64_t auto_nfft(int64_t nv, bool f64) {
    const int64_t nmax = f64 ? 8192 : 16384;
    int64_t best = 0;
    double best_cost = 0;
    for (int64_t n = 1024; n <= nmax; n <<= 1) {
        if (n - nv + 1 < n / 2) continue;   // at least half of every block must be new output
        const double cost = (double)n * (log2((double)n) + 2.0) / (double)(n - nv + 1);
        if (best == 0 || cost < best_cost) { best = n; best_cost = cost; }
    }
    if (best) return best;
    int64_t n = 4096;
    while (n < 4 * nv) n <<= 1;   // generic path: 75 % of each block is new output
    return n;
}

static int ensure_streams(OsPlanImpl* p) {
    if (p->s_exec) return DSPB200_OK;
    DSP_CUDA(cudaStreamCreateWithFlags(&p->s_in, cudaStreamNonBlocking));
    DSP_CUDA(cudaStreamCreateWithFlags(&p->s_exec, cudaStreamNonBlocking));
    DSP_CUDA(cudaStreamCreateWithFlags(&p->s_out, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        DSP_CUDA(cudaEventCreateWithFlags(&p->ev_in[i], cudaEventDisableTiming));
        DSP_CUDA(cudaEventCreateWithFlags(&p->ev_exec[i], cudaEventDisableTiming));
        DSP_CUDA(cudaEventCreateWithFlags(&p->ev_out[i], cudaEventDisableTiming));
    }
    return DSPB200_OK;
}

}  // namespace dspb200

using namespace dspb200;

struct dspb200_os_plan {
    OsPlanImpl impl;
};

// conv(u, v) for rank-2 / rank-3 arrays on device pointers: _conv_td! (mode 0), _conv_kern_fft! (mode 1: one N-D FFT pair of
// size nffts) or unsafe_conv_kern_os! (mode 2: blocks of nffts, batched).  Plans and scratch come from the cache / arena of
// runtime.cu; the caller holds the ConvenienceLock and synchronises the stream before the arena is reused.
enum { ND_DIRECT = 0, ND_FFT = 1, ND_OS = 2 };
static size_t g_nd_os_budget = (size_t)1 << 30;          // bytes of block buffers per batch (dspb200_conv_nd_os_* entry points)

template <typename T, bool CPLX>
static int conv_nd_dev(int mode, int rank, const int64_t* usize, const void* d_u, const int64_t* vsize, const void* d_v,
                       const int64_t* nffts, void* d_out, cudaStream_t st) {
    using E = typename os_elt<T, CPLX>::type;
    Dims3 su{{1, 1, 1}}, sv{{1, 1, 1}}, so{{1, 1, 1}}, sf{{1, 1, 1}};
    for (int d = 0; d < rank; ++d) {
        su.n[d] = usize[d]; sv.n[d] = vsize[d]; so.n[d] = usize[d] + vsize[d] - 1;
        if (mode != ND_DIRECT) sf.n[d] = nffts[d];
    }
    const int64_t no = so.n[0] * so.n[1] * so.n[2];
    const int threads = 256;
    if (mode == ND_DIRECT) {
        conv_direct_nd_kernel<T, CPLX><<<grid_for(no, 128), 128, 0, st>>>(d_u, su, d_v, sv, d_out);
        DSP_LAUNCH_OK();
        return DSPB200_OK;
    }
    DevBuf &tu = scratch_buf(3), &fu = scratch_buf(4), &fv = scratch_buf(5);
    const int64_t nf = sf.n[0] * sf.n[1] * sf.n[2];
    Dims3 sb = sf;                                           // spectrum dims: first (fastest) dim halved for real input
    if (!CPLX) sb.n[0] = sf.n[0] / 2 + 1;
    const int64_t nb = sb.n[0] * sb.n[1] * sb.n[2];
    long long nn[3];                                         // cuFFT is row-major: slowest dimension first
    for (int d = 0; d < rank; ++d) nn[d] = (long long)sf.n[rank - 1 - d];
    const bool f64 = sizeof(T) == 8;
    const int tf = CPLX ? (f64 ? CUFFT_Z2Z : CUFFT_C2C) : (f64 ? CUFFT_D2Z : CUFFT_R2C);
    const int ti = CPLX ? tf : (f64 ? CUFFT_Z2D : CUFFT_C2R);
    OsPlanImpl tmp;
    tmp.cplx = CPLX; tmp.f64 = f64;
    E zero;
    if constexpr (CPLX) zero = mkc<T>(T(0), T(0)); else zero = T(0);
    int h1f = 0;
    DSP_TRY(plan_cache_get(&h1f, rank, nn, false, 0, 0, tf, 1));
    if (mode == ND_FFT) {
        int h1i = h1f;
        if (!CPLX) DSP_TRY(plan_cache_get(&h1i, rank, nn, false, 0, 0, ti, 1));
        DSP_TRY(tu.reserve((size_t)nf * sizeof(E)));
        DSP_TRY(fu.reserve((size_t)nb * sizeof(cx<T>))); DSP_TRY(fv.reserve((size_t)nb * sizeof(cx<T>)));
        nd_copy_kernel<E><<<grid_for(nf, threads), threads, 0, st>>>((const E*)d_u, su, (E*)tu.p, sf, zero);
        DSP_LAUNCH_OK();
        DSP_TRY(generic_exec_fwd(&tmp, (cufftHandle)h1f, tu.p, fu.p, st));
        nd_copy_kernel<E><<<grid_for(nf, threads), threads, 0, st>>>((const E*)d_v, sv, (E*)tu.p, sf, zero);
        DSP_LAUNCH_OK();
        DSP_TRY(generic_exec_fwd(&tmp, (cufftHandle)h1f, tu.p, fv.p, st));
        scale_cplx_kernel<T><<<grid_for(nb, threads), threads, 0, st>>>((cx<T>*)fv.p, nb, T(1) / (T)nf);
        os_cmul_kernel<T><<<grid_for(nb, threads), threads, 0, st>>>((cx<T>*)fu.p, (const cx<T>*)fv.p, nb, 1);
        count_launch(2);
        DSP_TRY(generic_exec_inv(&tmp, (cufftHandle)h1i, fu.p, tu.p, st));
        nd_copy_kernel<E><<<grid_for(no, threads), threads, 0, st>>>((const E*)tu.p, sf, (E*)d_out, so, zero);
        DSP_LAUNCH_OK();
        return DSPB200_OK;
    }
    // ND_OS
    OsNd g;
    int64_t nblocks = 1, Lp = 1;
    for (int d = 0; d < 3; ++d) {
        g.su[d] = su.n[d]; g.sv[d] = sv.n[d]; g.so[d] = so.n[d]; g.nf[d] = sf.n[d];
        const int64_t ideal = sf.n[d] - sv.n[d] + 1;                           // :500
        g.L[d] = ideal < so.n[d] ? ideal : so.n[d];                             // save_blocksize = ideal - sout_deficit, :503-505
        g.nb[d] = cdiv(so.n[d], g.L[d]);                                        // :506
        nblocks *= g.nb[d]; Lp *= g.L[d];
    }
    const size_t per_block = (size_t)nf * sizeof(E) + (size_t)nb * sizeof(cx<T>);
    int64_t batch = (int64_t)(g_nd_os_budget / per_block);
    if (batch < 1) batch = 1;
    if (batch > nblocks) batch = nblocks;
    int hbf = h1f, hbi = 0;
    if (batch > 1) DSP_TRY(plan_cache_get(&hbf, rank, nn, false, 0, 0, tf, batch));
    if (CPLX) hbi = hbf; else DSP_TRY(plan_cache_get(&hbi, rank, nn, false, 0, 0, ti, batch));
    DSP_TRY(tu.reserve((size_t)nf * batch * sizeof(E)));
    DSP_TRY(fu.reserve((size_t)nb * batch * sizeof(cx<T>))); DSP_TRY(fv.reserve((size_t)nb * sizeof(cx<T>)));
    // filter spectrum, scaled once by 1/prod(nffts) (:513-516)
    nd_copy_kernel<E><<<grid_for(nf, threads), threads, 0, st>>>((const E*)d_v, sv, (E*)tu.p, sf, zero);
    DSP_LAUNCH_OK();
    DSP_TRY(generic_exec_fwd(&tmp, (cufftHandle)h1f, tu.p, fv.p, st));
    scale_cplx_kernel<T><<<grid_for(nb, threads), threads, 0, st>>>((cx<T>*)fv.p, nb, T(1) / (T)nf);
    DSP_LAUNCH_OK();
    for (int64_t b0 = 0; b0 < nblocks; b0 += batch) {
        nd_os_gather_kernel<E><<<grid_for(nf * batch, threads), threads, 0, st>>>((const E*)d_u, g, b0, batch, (E*)tu.p, zero);
        DSP_LAUNCH_OK();
        DSP_TRY(generic_exec_fwd(&tmp, (cufftHandle)hbf, tu.p, fu.p, st));
        os_cmul_kernel<T><<<grid_for(nb * batch, threads), threads, 0, st>>>((cx<T>*)fu.p, (const cx<T>*)fv.p, nb, batch);
        DSP_LAUNCH_OK();
        DSP_TRY(generic_exec_inv(&tmp, (cufftHandle)hbi, fu.p, tu.p, st));
        nd_os_scatter_kernel<E><<<grid_for(Lp * batch, threads), threads, 0, st>>>((const E*)tu.p, g, b0, batch, (E*)d_out);
        DSP_LAUNCH_OK();
    }
    return DSPB200_OK;
}

static int conv_nd_check(int dtype, int mode, int rank, const int64_t* usize, const void* u, const int64_t* vsize, const void* v,
                         const int64_t* nffts, void* out) {
    DSP_REQUIRE(dtype_valid(dtype), "invalid dtype %d", dtype);
    DSP_REQUIRE(rank >= 1 && rank <= 3, "rank must be 1, 2 or 3");
    DSP_REQUIRE(usize && vsize && u && v && out, "NULL argument");
    DSP_REQUIRE(mode == ND_DIRECT || nffts, "nffts is NULL");
    for (int d = 0; d < rank; ++d) {
        DSP_REQUIRE(usize[d] >= 1 && vsize[d] >= 1, "empty input");
        if (mode == ND_FFT)
            DSP_REQUIRE(nffts[d] >= usize[d] + vsize[d] - 1 && nffts[d] < (int64_t(1) << 31), "nffts must cover the full output");
        if (mode == ND_OS)
            DSP_REQUIRE(nffts[d] >= vsize[d] && nffts[d] < (int64_t(1) << 31), "overlap-save nffts must be at least size(v)");
    }
    return DSPB200_OK;
}

static int conv_nd_dispatch(int dtype, int mode, int rank, const int64_t* usize, const void* d_u, const int64_t* vsize,
                            const void* d_v, const int64_t* nffts, void* d_out, cudaStream_t st) {
    switch (dtype) {
        case DSPB200_F32: return conv_nd_dev<float, false>(mode, rank, usize, d_u, vsize, d_v, nffts, d_out, st);
        case DSPB200_F64: return conv_nd_dev<double, false>(mode, rank, usize, d_u, vsize, d_v, nffts, d_out, st);
        case DSPB200_C32: return conv_nd_dev<float, true>(mode, rank, usize, d_u, vsize, d_v, nffts, d_out, st);
        default: return conv_nd_dev<double, true>(mode, rank, usize, d_u, vsize, d_v, nffts, d_out, st);
    }
}

// device-pointer form: returns after the work on `stream` has completed (the cached plans and the arena are shared)
static int conv_nd_run_dev(int dtype, int mode, int rank, const int64_t* usize, const void* d_u, const int64_t* vsize, const void* d_v,
                           const int64_t* nffts, void* d_out, cudaStream_t st) {
    ConvenienceLock lock;
    int rc = conv_nd_dispatch(dtype, mode, rank, usize, d_u, vsize, d_v, nffts, d_out, st);
    if (rc == DSPB200_OK) {
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize", __FILE__, __LINE__);
    } else {
        cudaStreamSynchronize(st);
    }
    scratch_trim((size_t)256 << 20);                             // plans and small buffers stay cached for the next call
    return rc;
}

// host-pointer form
static int conv_nd_run_host(int dtype, int mode, int rank, const int64_t* usize, const void* u, const int64_t* vsize, const void* v,
                            const int64_t* nffts, void* out) {
    int64_t nu = 1, nv = 1, no = 1;
    for (int d = 0; d < rank; ++d) { nu *= usize[d]; nv *= vsize[d]; no *= usize[d] + vsize[d] - 1; }
    const size_t esz = dtype_size(dtype);
    ConvenienceLock lock;
    DevBuf &du = scratch_buf(0), &dv = scratch_buf(1), &dout = scratch_buf(2);
    auto body = [&]() -> int {
        DSP_TRY(du.reserve((size_t)nu * esz)); DSP_TRY(dv.reserve((size_t)nv * esz)); DSP_TRY(dout.reserve((size_t)no * esz));
        DSP_CUDA(cudaMemcpy(du.p, u, (size_t)nu * esz, cudaMemcpyHostToDevice));
        DSP_CUDA(cudaMemcpy(dv.p, v, (size_t)nv * esz, cudaMemcpyHostToDevice));
        DSP_TRY(conv_nd_dispatch(dtype, mode, rank, usize, du.p, vsize, dv.p, nffts, dout.p, 0));
        DSP_CUDA(cudaMemcpy(out, dout.p, (size_t)no * esz, cudaMemcpyDeviceToHost));
        return DSPB200_OK;
    };
    const int rc = body();
    if (rc != DSPB200_OK) cudaDeviceSynchronize();
    scratch_trim((size_t)256 << 20);
    return rc;
}

extern "C" {

int dspb200_os_plan_create(dspb200_os_plan** plan, int dtype, const void* v_host, int64_t nv, int64_t nfft) {
    DSP_RANGE("dspb200_os_plan_create");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    *plan = nullptr;
    DSP_REQUIRE(dtype_valid(dtype), "invalid dtype %d", dtype);
    DSP_REQUIRE(v_host != nullptr && nv >= 1, "filter must be non-empty");
    DSP_REQUIRE(nfft == 0 || nfft >= nv, "nfft (%lld) must be >= nv (%lld)", (long long)nfft, (long long)nv);
    DSP_REQUIRE(nfft < (int64_t(1) << 30), "nfft too large");
    dspb200_os_plan* h = new (std::nothrow) dspb200_os_plan();
    DSP_REQUIRE(h != nullptr, "out of host memory");
    OsPlanImpl* p = &h->impl;
    p->dtype = dtype; p->cplx = dtype_is_cplx(dtype); p->f64 = dtype_is_f64(dtype);
    p->nv = nv;
    p->nfft = nfft ? nfft : auto_nfft(nv, p->f64);
    p->L = p->nfft - nv + 1;
    p->fused = os_fused_ok(p->nfft, nv, p->f64);
    const size_t esz = dtype_size(dtype), csz = p->f64 ? 16 : 8;
    int rc = DSPB200_OK;
    void* d_v = nullptr;
    do {
        cudaError_t e = cudaGetDevice(&p->device);
        if (e == cudaSuccess) e = cudaMalloc(&d_v, (size_t)nv * esz);
        if (e == cudaSuccess) e = cudaMemcpy(d_v, v_host, (size_t)nv * esz, cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { rc = cuda_fail(e, "filter upload", __FILE__, __LINE__); break; }
        if (p->fused) {
            std::vector<unsigned char> tw((size_t)(fft_tl_len_rt(p->nfft) + 1) * csz), t16((size_t)fft_tw16_len(p->nfft) * csz), t256((size_t)fft_tw256_len(p->nfft) * csz);
            if (p->f64) {
                fft_fill_tl<double>((cx<double>*)tw.data(), p->nfft);
                fft_fill_tables<double>((cx<double>*)t16.data(), (cx<double>*)t256.data(), p->nfft);
            } else {
                fft_fill_tl<float>((cx<float>*)tw.data(), p->nfft);
                fft_fill_tables<float>((cx<float>*)t16.data(), (cx<float>*)t256.data(), p->nfft);
            }
            p->sm_count = device_sm_count();
            e = cudaMalloc(&p->d_tw, tw.size());
            if (e == cudaSuccess) e = cudaMemcpy(p->d_tw, tw.data(), tw.size(), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc(&p->d_t16, t16.size());
            if (e == cudaSuccess) e = cudaMemcpy(p->d_t16, t16.data(), t16.size(), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc(&p->d_t256, t256.size());
            if (e == cudaSuccess) e = cudaMemcpy(p->d_t256, t256.data(), t256.size(), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMalloc(&p->d_H, (size_t)p->nfft * csz);
            if (e == cudaSuccess && !p->f64 && p->nfft == 16384) {             // tables of the 32 x 32 x 16 kernel
                std::vector<cx<float>> a32(r32::T32_LEN), a1024(r32::T1024_LEN);
                r32::fill_tables<float>(a32.data(), a1024.data());
                e = cudaMalloc(&p->d_t32, a32.size() * sizeof(cx<float>));
                if (e == cudaSuccess) e = cudaMemcpy(p->d_t32, a32.data(), a32.size() * sizeof(cx<float>), cudaMemcpyHostToDevice);
                if (e == cudaSuccess) e = cudaMalloc(&p->d_t1024, a1024.size() * sizeof(cx<float>));
                if (e == cudaSuccess) e = cudaMemcpy(p->d_t1024, a1024.data(), a1024.size() * sizeof(cx<float>), cudaMemcpyHostToDevice);
            }
            if (e != cudaSuccess) { rc = cuda_fail(e, "twiddle upload", __FILE__, __LINE__); break; }
            rc = p->f64 ? os_filter_dispatch<double>(p, d_v) : os_filter_dispatch<float>(p, d_v);
        } else {
            p->nbins = p->cplx ? p->nfft : p->nfft / 2 + 1;
            int64_t b = (int64_t(1) << 22) / p->nfft;   // ~32 MiB (C32) of blocks in flight: stays L2-resident
            if (b < 1) b = 1;
            if (b > 4096) b = 4096;
            p->batch = b;
            rc = make_plans(p->cplx, p->f64, p->nfft, b, &p->fwd, &p->inv);
            if (rc != DSPB200_OK) break;
            p->fft_ok = true;
            rc = p->td.reserve((size_t)(b * p->nfft) * esz);
            if (rc == DSPB200_OK) rc = p->fd.reserve((size_t)(b * p->nbins) * csz);
            if (rc != DSPB200_OK) break;
            e = cudaMalloc(&p->d_H, (size_t)p->nbins * csz);
            if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMalloc(H)", __FILE__, __LINE__); break; }
            // H = FFT(zero-padded v / nfft): reuse the batch plan on row 0 of td (other rows zero)
            e = cudaMemset(p->td.p, 0, (size_t)(b * p->nfft) * esz);
            if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemset", __FILE__, __LINE__); break; }
            const int threads = 256;
            if (p->f64) {
                if (p->cplx) pad_copy_kernel<double, true><<<grid_for(p->nfft, threads), threads>>>(d_v, nv, p->td.p, p->nfft, 1.0 / (double)p->nfft);
                else pad_copy_kernel<double, false><<<grid_for(p->nfft, threads), threads>>>(d_v, nv, p->td.p, p->nfft, 1.0 / (double)p->nfft);
            } else {
                if (p->cplx) pad_copy_kernel<float, true><<<grid_for(p->nfft, threads), threads>>>(d_v, nv, p->td.p, p->nfft, 1.0f / (float)p->nfft);
                else pad_copy_kernel<float, false><<<grid_for(p->nfft, threads), threads>>>(d_v, nv, p->td.p, p->nfft, 1.0f / (float)p->nfft);
            }
            count_launch(1);
            rc = generic_exec_fwd(p, p->fwd, p->td.p, p->fd.p, 0);
            if (rc != DSPB200_OK) break;
            e = cudaMemcpy(p->d_H, p->fd.p, (size_t)p->nbins * csz, cudaMemcpyDeviceToDevice);
            if (e == cudaSuccess) e = cudaDeviceSynchronize();
            if (e != cudaSuccess) { rc = cuda_fail(e, "filter transform", __FILE__, __LINE__); break; }
        }
    } while (0);
    if (d_v) cudaFree(d_v);
    if (rc != DSPB200_OK) { dspb200_os_plan_destroy(h); return rc; }
    *plan = h;
    return DSPB200_OK;
}

int dspb200_os_plan_nfft(const dspb200_os_plan* plan, int64_t* nfft, int* fused) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    if (nfft) *nfft = plan->impl.nfft;
    if (fused) *fused = plan->impl.fused ? 1 : 0;
    return DSPB200_OK;
}

int dspb200_os_plan_geometry(const dspb200_os_plan* plan, int* dtype, int64_t* nv, int64_t* nfft) {
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    if (dtype) *dtype = plan->impl.dtype;
    if (nv) *nv = plan->impl.nv;
    if (nfft) *nfft = plan->impl.nfft;
    return DSPB200_OK;
}

int dspb200_os_exec_dev(dspb200_os_plan* plan, const void* u, int64_t nu, int64_t ncols, void* out, int64_t nout,
                        void* stream) {
    DSP_RANGE("dspb200_os_exec_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nu >= 0 && ncols >= 0 && nout >= 0, "negative size");
    if (nout == 0 || ncols == 0) return DSPB200_OK;
    DSP_REQUIRE(out != nullptr && (u != nullptr || nu == 0), "NULL argument");
    OsPlanImpl* p = &plan->impl;
    if (nu == 0) {
        DSP_CUDA(cudaMemsetAsync(out, 0, (size_t)(nout * ncols) * dtype_size(p->dtype), (cudaStream_t)stream));
        return DSPB200_OK;
    }
    OsRange a{u, 0, nu, nu, out, 0, nout, nout, nu + p->nv - 1, ncols};
    return os_run(p, a, (cudaStream_t)stream);
}

int dspb200_os_exec_range_dev(dspb200_os_plan* plan, const void* u_local, int64_t u_begin, int64_t nu_local,
                              void* out_local, int64_t out_begin, int64_t out_count, void* stream) {
    DSP_RANGE("dspb200_os_exec_range_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nu_local >= 0 && out_count >= 0 && out_begin >= 0, "bad range");
    if (out_count == 0) return DSPB200_OK;
    DSP_REQUIRE(out_local != nullptr && (u_local != nullptr || nu_local == 0), "NULL argument");
    OsPlanImpl* p = &plan->impl;
    OsRange a{u_local, u_begin, nu_local, 0, out_local, out_begin, out_count, 0, INT64_MAX, 1};
    return os_run(p, a, (cudaStream_t)stream);
}

// Host pointers.  One long column is streamed: chunk c+1 is copied in while chunk c is convolved and chunk
// c-1 is copied out (three streams, two buffers each); otherwise copy in -> run -> copy out.
int dspb200_os_exec(dspb200_os_plan* plan, const void* u, int64_t nu, int64_t ncols, void* out, int64_t nout) {
    DSP_RANGE("dspb200_os_exec");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nu >= 0 && ncols >= 0 && nout >= 0, "negative size");
    if (nout == 0 || ncols == 0) return DSPB200_OK;
    DSP_REQUIRE(out != nullptr && (u != nullptr || nu == 0), "NULL argument");
    OsPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    DSP_TRY(ensure_streams(p));
    const size_t esz = dtype_size(p->dtype);
    const int64_t chunk_out = ((int64_t(32) << 20) / (int64_t)esz / p->L + 1) * p->L;   // ~32 MiB, whole blocks
    if (ncols == 1 && nout > 2 * chunk_out && nu > 0) {
        const int64_t nfull = nu + p->nv - 1;
        const size_t in_cap = (size_t)(chunk_out + p->nv - 1) * esz, out_cap = (size_t)chunk_out * esz;
        for (int i = 0; i < 2; ++i) { DSP_TRY(p->in[i].reserve(in_cap)); DSP_TRY(p->out[i].reserve(out_cap)); }
        bool used[2] = {false, false};
        int slot = 0;
        for (int64_t m0 = 0; m0 < nout; m0 += chunk_out, slot ^= 1) {
            const int64_t cnt = nout - m0 < chunk_out ? nout - m0 : chunk_out;
            int64_t i_lo = m0 - (p->nv - 1); if (i_lo < 0) i_lo = 0;
            int64_t i_hi = m0 + cnt; if (i_hi > nu) i_hi = nu;
            const int64_t ni = i_hi > i_lo ? i_hi - i_lo : 0;
            if (used[slot]) DSP_CUDA(cudaStreamWaitEvent(p->s_in, p->ev_exec[slot], 0));    // input buffer free
            if (ni > 0) DSP_CUDA(cudaMemcpyAsync(p->in[slot].p, (const char*)u + (size_t)i_lo * esz, (size_t)ni * esz, cudaMemcpyHostToDevice, p->s_in));
            DSP_CUDA(cudaEventRecord(p->ev_in[slot], p->s_in));
            DSP_CUDA(cudaStreamWaitEvent(p->s_exec, p->ev_in[slot], 0));
            if (used[slot]) DSP_CUDA(cudaStreamWaitEvent(p->s_exec, p->ev_out[slot], 0));  // output buffer drained
            OsRange a{p->in[slot].p, i_lo, ni, 0, p->out[slot].p, m0, cnt, 0, nfull, 1};
            DSP_TRY(os_run(p, a, p->s_exec));
            DSP_CUDA(cudaEventRecord(p->ev_exec[slot], p->s_exec));
            DSP_CUDA(cudaStreamWaitEvent(p->s_out, p->ev_exec[slot], 0));
            DSP_CUDA(cudaMemcpyAsync((char*)out + (size_t)m0 * esz, p->out[slot].p, (size_t)cnt * esz, cudaMemcpyDeviceToHost, p->s_out));
            DSP_CUDA(cudaEventRecord(p->ev_out[slot], p->s_out));
            used[slot] = true;
        }
        DSP_CUDA(cudaStreamSynchronize(p->s_out));
        DSP_CUDA(cudaStreamSynchronize(p->s_exec));
        return DSPB200_OK;
    }
    const size_t in_bytes = (size_t)(nu * ncols) * esz, out_bytes = (size_t)(nout * ncols) * esz;
    DSP_TRY(p->in[0].reserve(in_bytes ? in_bytes : 16));
    DSP_TRY(p->out[0].reserve(out_bytes));
    if (in_bytes) DSP_CUDA(cudaMemcpyAsync(p->in[0].p, u, in_bytes, cudaMemcpyHostToDevice, p->s_exec));
    DSP_TRY(dspb200_os_exec_dev(plan, p->in[0].p, nu, ncols, p->out[0].p, nout, p->s_exec));
    DSP_CUDA(cudaMemcpyAsync(out, p->out[0].p, out_bytes, cudaMemcpyDeviceToHost, p->s_exec));
    DSP_CUDA(cudaStreamSynchronize(p->s_exec));
    return DSPB200_OK;
}

int dspb200_os_plan_destroy(dspb200_os_plan* plan) {
    if (!plan) return DSPB200_OK;
    OsPlanImpl* p = &plan->impl;
    if (p->d_tw) cudaFree(p->d_tw);
    if (p->d_t16) cudaFree(p->d_t16);
    if (p->d_t256) cudaFree(p->d_t256);
    if (p->d_t32) cudaFree(p->d_t32);
    if (p->d_t1024) cudaFree(p->d_t1024);
    if (p->d_H) cudaFree(p->d_H);
    if (p->fft_ok) { cufftDestroy(p->fwd); cufftDestroy(p->inv); }
    p->td.release(); p->fd.release();
    for (int i = 0; i < 2; ++i) {
        p->in[i].release(); p->out[i].release();
        if (p->ev_in[i]) cudaEventDestroy(p->ev_in[i]);
        if (p->ev_exec[i]) cudaEventDestroy(p->ev_exec[i]);
        if (p->ev_out[i]) cudaEventDestroy(p->ev_out[i]);
    }
    if (p->s_in) cudaStreamDestroy(p->s_in);
    if (p->s_exec) cudaStreamDestroy(p->s_exec);
    if (p->s_out) cudaStreamDestroy(p->s_out);
    delete plan;
    return DSPB200_OK;
}

// _conv_kern_fft!, src/dspbase.jl:611-644 (host pointers; cuFFT plans and scratch from the process-wide cache)
int dspb200_conv_fft_exec(int dtype, const void* u, int64_t nu, const void* v, int64_t nv, int64_t nfft, void* out) {
    DSP_RANGE("dspb200_conv_fft_exec");
    DSP_REQUIRE(dtype_valid(dtype), "invalid dtype %d", dtype);
    DSP_REQUIRE(u && v && out && nu >= 1 && nv >= 1, "empty or NULL input");
    const int64_t nout = nu + nv - 1;
    DSP_REQUIRE(nfft >= nout, "nfft (%lld) must be >= nu+nv-1 (%lld)", (long long)nfft, (long long)nout);
    DSP_REQUIRE(nfft < (int64_t(1) << 31), "nfft too large");
    OsPlanImpl tmp;
    tmp.dtype = dtype; tmp.cplx = dtype_is_cplx(dtype); tmp.f64 = dtype_is_f64(dtype);
    const size_t esz = dtype_size(dtype), csz = tmp.f64 ? 16 : 8;
    const int64_t nbins = tmp.cplx ? nfft : nfft / 2 + 1;
    ConvenienceLock lock;                                       // cached plans + scratch arena (common.cuh)
    DevBuf &du = scratch_buf(0), &dv = scratch_buf(1), &tu = scratch_buf(3), &fu = scratch_buf(4), &fv = scratch_buf(5);
    cufftHandle fwd = 0, inv = 0;
    int rc = DSPB200_OK;
    auto body = [&]() -> int {
        DSP_TRY(du.reserve((size_t)nu * esz)); DSP_TRY(dv.reserve((size_t)nv * esz));
        DSP_TRY(tu.reserve((size_t)nfft * esz));
        DSP_TRY(fu.reserve((size_t)nbins * csz)); DSP_TRY(fv.reserve((size_t)nbins * csz));
        DSP_CUDA(cudaMemcpy(du.p, u, (size_t)nu * esz, cudaMemcpyHostToDevice));
        DSP_CUDA(cudaMemcpy(dv.p, v, (size_t)nv * esz, cudaMemcpyHostToDevice));
        {
            long long nn[1] = {(long long)nfft};
            int hf = 0, hi = 0;
            if (tmp.cplx) {
                DSP_TRY(plan_cache_get(&hf, 1, nn, false, 0, 0, tmp.f64 ? CUFFT_Z2Z : CUFFT_C2C, 1));
                hi = hf;
            } else {
                DSP_TRY(plan_cache_get(&hf, 1, nn, false, 0, 0, tmp.f64 ? CUFFT_D2Z : CUFFT_R2C, 1));
                DSP_TRY(plan_cache_get(&hi, 1, nn, false, 0, 0, tmp.f64 ? CUFFT_Z2D : CUFFT_C2R, 1));
            }
            fwd = (cufftHandle)hf; inv = (cufftHandle)hi;
        }
        const int threads = 256;
        const int g = grid_for(nfft, threads);
#define PAD(SRC, N_) \
        if (tmp.f64) { if (tmp.cplx) pad_copy_kernel<double, true><<<g, threads>>>(SRC, N_, tu.p, nfft, 1.0); else pad_copy_kernel<double, false><<<g, threads>>>(SRC, N_, tu.p, nfft, 1.0); } \
        else { if (tmp.cplx) pad_copy_kernel<float, true><<<g, threads>>>(SRC, N_, tu.p, nfft, 1.0f); else pad_copy_kernel<float, false><<<g, threads>>>(SRC, N_, tu.p, nfft, 1.0f); } \
        count_launch(1);
        PAD(du.p, nu)
        DSP_TRY(generic_exec_fwd(&tmp, fwd, tu.p, fu.p, 0));
        PAD(dv.p, nv)
        DSP_TRY(generic_exec_fwd(&tmp, fwd, tu.p, fv.p, 0));
#undef PAD
        // fv *= 1/nfft ; fu *= fv
        if (tmp.f64) {
            scale_cplx_kernel<double><<<grid_for(nbins, threads), threads>>>((cx<double>*)fv.p, nbins, 1.0 / (double)nfft);
            os_cmul_kernel<double><<<grid_for(nbins, threads), threads>>>((cx<double>*)fu.p, (const cx<double>*)fv.p, nbins, 1);
        } else {
            scale_cplx_kernel<float><<<grid_for(nbins, threads), threads>>>((cx<float>*)fv.p, nbins, 1.0f / (float)nfft);
            os_cmul_kernel<float><<<grid_for(nbins, threads), threads>>>((cx<float>*)fu.p, (const cx<float>*)fv.p, nbins, 1);
        }
        count_launch(2);
        DSP_TRY(generic_exec_inv(&tmp, inv, fu.p, tu.p, 0));
        DSP_CUDA(cudaMemcpy(out, tu.p, (size_t)nout * esz, cudaMemcpyDeviceToHost));
        return DSPB200_OK;
    };
    rc = body();
    scratch_trim((size_t)256 << 20);
    return rc;
}

// conv(u, v) / conv!(out, u, v) for matrices and rank-3 arrays, src/dspbase.jl:611-660, 709-757 (cached plans)
int dspb200_conv_nd_exec(int dtype, int rank, const int64_t* usize, const void* u, const int64_t* vsize, const void* v,
                         const int64_t* nffts, void* out) {
    DSP_RANGE("dspb200_conv_nd_exec");
    const int mode = nffts ? ND_FFT : ND_DIRECT;
    DSP_TRY(conv_nd_check(dtype, mode, rank, usize, u, vsize, v, nffts, out));
    return conv_nd_run_host(dtype, mode, rank, usize, u, vsize, v, nffts, out);
}
int dspb200_conv_nd_exec_dev(int dtype, int rank, const int64_t* usize, const void* d_u, const int64_t* vsize, const void* d_v,
                             const int64_t* nffts, void* d_out, void* stream) {
    DSP_RANGE("dspb200_conv_nd_exec_dev");
    const int mode = nffts ? ND_FFT : ND_DIRECT;
    DSP_TRY(conv_nd_check(dtype, mode, rank, usize, d_u, vsize, d_v, nffts, d_out));
    return conv_nd_run_dev(dtype, mode, rank, usize, d_u, vsize, d_v, nffts, d_out, reinterpret_cast<cudaStream_t>(stream));
}

// conv(u, v; algorithm=:fft_overlapsave) for arrays of rank <= 3: unsafe_conv_kern_os!, src/dspbase.jl:371-609
int dspb200_conv_nd_os_exec(int dtype, int rank, const int64_t* usize, const void* u, const int64_t* vsize, const void* v,
                            const int64_t* nffts, void* out) {
    DSP_RANGE("dspb200_conv_nd_os_exec");
    DSP_TRY(conv_nd_check(dtype, ND_OS, rank, usize, u, vsize, v, nffts, out));
    return conv_nd_run_host(dtype, ND_OS, rank, usize, u, vsize, v, nffts, out);
}
int dspb200_conv_nd_os_exec_dev(int dtype, int rank, const int64_t* usize, const void* d_u, const int64_t* vsize, const void* d_v,
                                const int64_t* nffts, void* d_out, void* stream) {
    DSP_RANGE("dspb200_conv_nd_os_exec_dev");
    DSP_TRY(conv_nd_check(dtype, ND_OS, rank, usize, d_u, vsize, d_v, nffts, d_out));
    return conv_nd_run_dev(dtype, ND_OS, rank, usize, d_u, vsize, d_v, nffts, d_out, reinterpret_cast<cudaStream_t>(stream));
}
int dspb200_conv_nd_os_set_budget(size_t bytes) {
    DSP_REQUIRE(bytes >= 1, "the block-buffer budget must be positive");
    g_nd_os_budget = bytes;
    return DSPB200_OK;
}

// hilbert(x), src/util.jl:31-75 (kernel: hilbert_weight_kernel above)
int dspb200_hilbert_exec_dev(int dtype, const void* d_x, int64_t n, int64_t ncols, void* d_out, void* stream) {
    DSP_RANGE("dspb200_hilbert_exec_dev");
    DSP_REQUIRE(dtype == DSPB200_F32 || dtype == DSPB200_F64, "hilbert takes a real signal (dtype %d)", dtype);
    DSP_REQUIRE(d_x && d_out && n >= 1 && ncols >= 1, "empty or NULL input");
    DSP_REQUIRE(n < (int64_t(1) << 31), "n too large");
    const bool f64 = dtype == DSPB200_F64;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    cufftHandle fwd = 0, inv = 0;
    ConvenienceLock lock;                                       // cached plans (common.cuh)
    auto body = [&]() -> int {
        long long nn[1] = {(long long)n};
        int hf = 0, hi = 0;
        // real -> complex, column c: n reals at c*n  ->  n/2+1 bins at the start of the n-bin output column c
        DSP_TRY(plan_cache_get(&hf, 1, nn, true, n, n, f64 ? CUFFT_D2Z : CUFFT_R2C, ncols));
        DSP_TRY(plan_cache_get(&hi, 1, nn, false, 0, 0, f64 ? CUFFT_Z2Z : CUFFT_C2C, ncols));
        fwd = (cufftHandle)hf; inv = (cufftHandle)hi;
        DSP_CUFFT(cufftSetStream(fwd, st));
        DSP_CUFFT(cufftSetStream(inv, st));
        const int threads = 256, g = grid_for(n * ncols, threads);
        if (f64) {
            DSP_CUFFT(cufftExecD2Z(fwd, (cufftDoubleReal*)const_cast<void*>(d_x), (cufftDoubleComplex*)d_out));
            hilbert_weight_kernel<double><<<g, threads, 0, st>>>((cx<double>*)d_out, n, ncols, 1.0 / (double)n);
            DSP_LAUNCH_OK();
            DSP_CUFFT(cufftExecZ2Z(inv, (cufftDoubleComplex*)d_out, (cufftDoubleComplex*)d_out, CUFFT_INVERSE));
        } else {
            DSP_CUFFT(cufftExecR2C(fwd, (cufftReal*)const_cast<void*>(d_x), (cufftComplex*)d_out));
            hilbert_weight_kernel<float><<<g, threads, 0, st>>>((cx<float>*)d_out, n, ncols, 1.0f / (float)n);
            DSP_LAUNCH_OK();
            DSP_CUFFT(cufftExecC2C(inv, (cufftComplex*)d_out, (cufftComplex*)d_out, CUFFT_INVERSE));
        }
        count_launch(2);
        DSP_CUDA(cudaStreamSynchronize(st));              // the cached plans may be re-targeted to another stream by the next call
        return DSPB200_OK;
    };
    return body();
}

int dspb200_hilbert_exec(int dtype, const void* x, int64_t n, int64_t ncols, void* out) {
    DSP_RANGE("dspb200_hilbert_exec");
    DSP_REQUIRE(dtype == DSPB200_F32 || dtype == DSPB200_F64, "hilbert takes a real signal (dtype %d)", dtype);
    DSP_REQUIRE(x && out && n >= 1 && ncols >= 1, "empty or NULL input");
    const size_t esz = dtype_size(dtype);
    DevBuf dx, dout;
    auto body = [&]() -> int {
        DSP_TRY(dx.reserve((size_t)(n * ncols) * esz));
        DSP_TRY(dout.reserve((size_t)(n * ncols) * 2 * esz));
        DSP_CUDA(cudaMemcpy(dx.p, x, (size_t)(n * ncols) * esz, cudaMemcpyHostToDevice));
        DSP_TRY(dspb200_hilbert_exec_dev(dtype, dx.p, n, ncols, dout.p, nullptr));
        DSP_CUDA(cudaMemcpy(out, dout.p, (size_t)(n * ncols) * 2 * esz, cudaMemcpyDeviceToHost));
        return DSPB200_OK;
    };
    const int rc = body();
    dx.release(); dout.release();
    return rc;
}

// _conv_td!, src/dspbase.jl:646-660 (host pointers)
int dspb200_conv_direct_exec(int dtype, const void* u, int64_t nu, const void* v, int64_t nv, void* out) {
    DSP_RANGE("dspb200_conv_direct_exec");
    DSP_REQUIRE(dtype_valid(dtype), "invalid dtype %d", dtype);
    DSP_REQUIRE(u && v && out && nu >= 1 && nv >= 1, "empty or NULL input");
    const size_t esz = dtype_size(dtype);
    const int64_t nout = nu + nv - 1;
    DevBuf du, dv, dout;
    auto body = [&]() -> int {
        DSP_TRY(du.reserve((size_t)nu * esz)); DSP_TRY(dv.reserve((size_t)nv * esz)); DSP_TRY(dout.reserve((size_t)nout * esz));
        DSP_CUDA(cudaMemcpy(du.p, u, (size_t)nu * esz, cudaMemcpyHostToDevice));
        DSP_CUDA(cudaMemcpy(dv.p, v, (size_t)nv * esz, cudaMemcpyHostToDevice));
        const void* large = nu >= nv ? du.p : dv.p;
        const void* small = nu >= nv ? dv.p : du.p;
        const int64_t nl = nu >= nv ? nu : nv, ns = nu >= nv ? nv : nu;
        const int threads = 128, g = grid_for(nout, threads);
        switch (dtype) {
            case DSPB200_F32: conv_direct_kernel<float, false><<<g, threads>>>(large, nl, small, ns, dout.p); break;
            case DSPB200_F64: conv_direct_kernel<double, false><<<g, threads>>>(large, nl, small, ns, dout.p); break;
            case DSPB200_C32: conv_direct_kernel<float, true><<<g, threads>>>(large, nl, small, ns, dout.p); break;
            default: conv_direct_kernel<double, true><<<g, threads>>>(large, nl, small, ns, dout.p); break;
        }
        DSP_LAUNCH_OK();
        DSP_CUDA(cudaMemcpy(out, dout.p, (size_t)nout * esz, cudaMemcpyDeviceToHost));
        return DSPB200_OK;
    };
    const int rc = body();
    du.release(); dv.release(); dout.release();
    return rc;
}

}  // extern "C"
