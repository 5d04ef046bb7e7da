// dspb200 -- rational / integer polyphase resampling: resample(x, rate, h) with rate = interp // decim.
//
// Reference path: FIRRational / FIRInterpolator / FIRDecimator kernels and their serial filt! loops
// (src/Filters/stream_filt.jl:8-78, 431-560), taps2pfb (:294-307), _resample! (:696-725).
// The (inputIdx, phiIdx) recurrence has the closed form (SURVEY.md App. A9)
//     p = phi0 + j*decim,  n = n0 + p / interp,  phi = p % interp,
//     y[j] = sum_{r=0..T-1} pfb[r, phi] * x[n - (T-1) + r]          (T = taps per phase)
// with pfb[r, phi] = hp[phi + (T-1-r)*interp] (each column reversed, :294-307), so every output sample is
// independent.  The dot product runs oldest sample first like unsafe_dot (src/util.jl:225-255), in the promoted
// eltype (:654).  Input samples outside the stored range are zero (zero history, :175, and _zeropad, :699).
//
// Layout: CTA = 256 outputs.  The polyphase bank is staged in shared memory phase-major when it fits;
// x is read through L1/L2 (neighbouring outputs share all but a few samples).
//
// rs_launch tries four kernels in order, each covering shapes the previous one cannot: resample_mp2_kernel (pipelined,
// interp <= 4, decim <= 4, at most 64 taps per phase) -> resample_mp_kernel -> resample_tiled_kernel -> resample_kernel.
// The pipelined kernel's configuration (4 outputs per phase per thread in Float32, packed FFMA2 for ComplexF32 samples,
// 128-bit tap loads, the rs_v3 tap rows) is the one that won the resample A/Bs in profiles/README.md; measured in round 2
// with variants since removed; see the history before this commit.
#include "common.cuh"
#include <cuda_pipeline.h>
#include <new>
#include <vector>

namespace dspb200 {

constexpr int RS_NT = 256;

template <typename TO, typename TX> struct rs_cvt;
template <typename TR> struct rs_cvt<TR, float>  { __device__ static __forceinline__ TR get(float v) { return (TR)v; } };
template <typename TR> struct rs_cvt<TR, double> { __device__ static __forceinline__ TR get(double v) { return (TR)v; } };
template <typename TR, typename S> struct rs_cvt<cx<TR>, cx<S>> { __device__ static __forceinline__ cx<TR> get(cx<S> v) { return mkc<TR>((TR)v.x, (TR)v.y); } };

template <typename TR> __device__ __forceinline__ TR rs_fma(TR h, TR x, TR acc) { return fma(h, x, acc); }
template <typename TR> __device__ __forceinline__ cx<TR> rs_fma(TR h, cx<TR> x, cx<TR> acc) {
    return mkc<TR>(fma(h, x.x, acc.x), fma(h, x.y, acc.y));
}
// real tap x ComplexF32 sample: both halves in ONE packed FFMA2 (sm_100: two IEEE fused multiply-adds per instruction, the
// tap broadcast to both halves) -- the same two roundings as the scalar pair, half the issue slots.
template <> __device__ __forceinline__ cx<float> rs_fma<float>(float h, cx<float> x, cx<float> acc) {
    const float2 r = __ffma2_rn(make_float2(h, h), make_float2(x.x, x.y), make_float2(acc.x, acc.y));
    return mkc<float>(r.x, r.y);
}
template <typename T> __device__ __forceinline__ T rs_zero(T*) { return T(0); }
template <typename T> __device__ __forceinline__ cx<T> rs_zero(cx<T>*) { return mkc<T>(T(0), T(0)); }

// EX: input element, TR: real arithmetic type, EO: output element (TR or cx<TR>)
template <typename EX, typename TR, typename EO>
__global__ void __launch_bounds__(RS_NT)
resample_kernel(const EX* __restrict__ x, int64_t x_begin, int64_t nx_local, int64_t x_col_stride,
                const TR* __restrict__ pfb /* [interp][tpp], accumulation order */, int tpp, int64_t interp,
                int64_t decim, int64_t n0, int64_t phi0, EO* __restrict__ out, int64_t j_begin, int64_t nout_local,
                int64_t out_col_stride, int64_t tiles_per_col, int pfb_in_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TR* ps = reinterpret_cast<TR*>(smem_raw);
    const int64_t col = blockIdx.x / tiles_per_col;
    const int64_t tile = blockIdx.x % tiles_per_col;
    if (pfb_in_smem) {
        const int64_t tot = interp * tpp;
        for (int64_t i = threadIdx.x; i < tot; i += RS_NT) ps[i] = pfb[i];
        __syncthreads();
    }
    const TR* bank = pfb_in_smem ? ps : pfb;
    const int64_t jl = tile * RS_NT + threadIdx.x;
    if (jl >= nout_local) return;
    const int64_t j = j_begin + jl;
    const int64_t p = phi0 + j * decim;
    const int64_t n = n0 + p / interp;
    const int64_t phi = p % interp;
    const TR* hcol = bank + phi * tpp;
    const EX* xc = x + col * x_col_stride;
    const int64_t first = n - (tpp - 1) - x_begin;   // local index of the oldest sample
    EO acc = rs_zero((EO*)nullptr);
    if (first >= 0 && first + tpp <= nx_local) {
        const EX* xp = xc + first;
        for (int r = 0; r < tpp; ++r) acc = rs_fma(hcol[r], rs_cvt<EO, EX>::get(xp[r]), acc);
    } else {
        for (int r = 0; r < tpp; ++r) {
            const int64_t i = first + r;
            if (i >= 0 && i < nx_local) acc = rs_fma(hcol[r], rs_cvt<EO, EX>::get(xc[i]), acc);
        }
    }
    out[col * out_col_stride + jl] = acc;
}

// ---------------------------------------------------------------------------------------------- register-tiled kernel
// For small decimation D (compile time) every thread computes G outputs of ONE phase (j, j+I, .., j+(G-1)I: same taps,
// inputs D apart), eight taps at a time: the (G-1)*D + 8 input samples those G x 8 products touch are loaded from the
// shared-memory tile once into registers and the tap chunk is loaded once, so the inner loop is G*8 multiply-adds per
// (G-1)*D + 8 + 2 shared loads (3//2, G = 8: 128 FFMA-pairs per 24 loads) -- FMA-bound instead of load-bound.
// CTA: I * MT threads = (phase slot i, time index m); outputs j0 + i + I*(G*m + g).  The x tile and the phase-major
// tap bank (rows padded with zeros to a multiple of 8) are staged in shared memory; results go back through shared
// memory so the global store is fully coalesced.  Same accumulation order as resample_kernel (oldest sample first).
template <typename EX, typename TR, typename EO, int D, int G>
__global__ void __launch_bounds__(256)
resample_tiled_kernel(const EX* __restrict__ x, int64_t x_begin, int64_t nx_local, int64_t x_col_stride,
                      const TR* __restrict__ pfb8 /* [interp][tpp8] */, int tpp, int tpp8, int interp, int mt,
                      int64_t n0, int64_t phi0, EO* __restrict__ out, int64_t j_begin, int64_t nout_local,
                      int64_t out_col_stride, int xtile_len) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TR* bank = reinterpret_cast<TR*>(smem_raw);                                   // interp * tpp8
    EX* xs = reinterpret_cast<EX*>(bank + (size_t)interp * tpp8);                 // xtile_len (+ slack)
    EO* os = reinterpret_cast<EO*>(xs);                                           // reused for the output tile
    __shared__ int64_t s_qt;                                                      // (phi0 + j0*D) div / mod interp
    __shared__ int s_rt;
    const int tid = threadIdx.x;
    const int nthreads = blockDim.x;
    const int64_t col = blockIdx.y;                                               // grid = (tiles, columns)
    const int64_t tile = blockIdx.x;
    const int tile_out = interp * G * mt;
    const int64_t jl0 = tile * tile_out;                                          // first local output of the tile
    const int64_t j0 = j_begin + jl0;
    // all 64-bit index arithmetic is per-CTA: one thread splits p_tile = phi0 + j0*D = interp*qt + rt; per-thread
    // offsets inside the tile then need only 32-bit divisions
    if (tid == 0) {
        const int64_t pt = phi0 + j0 * D;
        s_qt = pt / interp;
        s_rt = (int)(pt - (pt / interp) * interp);
    }
    for (int i = tid; i < interp * tpp8; i += nthreads) bank[i] = pfb8[i];
    __syncthreads();
    const int64_t qt = s_qt;
    const int rt = s_rt;
    // x range of the tile: oldest sample of its first output .. newest sample of its last output (+ chunk slack)
    const int64_t gb = n0 + qt - (tpp - 1) - x_begin;                             // local index of tile element 0
    const EX* xb = x + col * x_col_stride + gb;
    const int64_t lo64 = -gb, hi64 = nx_local - gb;
    const int i_lo = lo64 < 0 ? 0 : (lo64 > xtile_len ? xtile_len : (int)lo64);
    const int i_hi = hi64 < 0 ? 0 : (hi64 > xtile_len ? xtile_len : (int)hi64);
    for (int i = tid; i < xtile_len; i += nthreads) xs[i] = (i >= i_lo && i < i_hi) ? xb[i] : rs_zero((EX*)nullptr);
    __syncthreads();

    const int i_ph = tid % interp;
    const int m = tid / interp;
    EO acc[G];
#pragma unroll
    for (int g = 0; g < G; ++g) acc[g] = rs_zero((EO*)nullptr);
    const bool active = m < mt;
    if (active) {
        const int prel = rt + (i_ph + interp * G * m) * D;                        // p - interp*qt of its first output
        const int off = prel / interp;                                            // tile index of its oldest sample
        const int phi = prel - off * interp;
        const TR* hrow = bank + (size_t)phi * tpp8;
        for (int r0 = 0; r0 < tpp8; r0 += 8) {
            TR h[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) h[q] = hrow[r0 + q];
            EO xv[(G - 1) * D + 8];
#pragma unroll
            for (int q = 0; q < (G - 1) * D + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xs[off + r0 + q]);
            if (r0 + 8 <= tpp) {
#pragma unroll
                for (int q = 0; q < 8; ++q)
#pragma unroll
                    for (int g = 0; g < G; ++g) acc[g] = rs_fma(h[q], xv[g * D + q], acc[g]);
            } else {                       // last, partial chunk: the padding taps never touch a sample
#pragma unroll
                for (int q = 0; q < 8; ++q)
                    if (r0 + q < tpp) {
#pragma unroll
                        for (int g = 0; g < G; ++g) acc[g] = rs_fma(h[q], xv[g * D + q], acc[g]);
                    }
            }
        }
    }
    __syncthreads();                                                              // x tile no longer needed
    if (active) {
#pragma unroll
        for (int g = 0; g < G; ++g) os[i_ph + interp * (G * m + g)] = acc[g];
    }
    __syncthreads();
    EO* oc = out + col * out_col_stride + jl0;
    const int64_t remain = nout_local - jl0;
    const int cnt = remain < tile_out ? (int)remain : tile_out;
    for (int i = tid; i < cnt; i += nthreads) oc[i] = os[i];
}

// ---------------------------------------------------------------------------------------------- multi-phase tiled kernel
// Small interpolation factors (I <= 4, e.g. BASELINE config 5: 3//2).  The tiled kernel above gives a thread G outputs of
// ONE phase; per 8-tap chunk it loads (G-1)*D + 8 samples for G*8 products and is bound by shared-memory bandwidth
// (ncu, 3//2 ComplexF32: the LSU data pipe is the busiest unit, the FMA pipe ~25 %).  Here a thread computes I*G CONSECUTIVE
// outputs -- G of each of the I phases: their sample windows overlap almost completely (consecutive outputs advance by D/I
// samples), so the same (I*G-1)*D/I + 8 samples feed I*G*8 products: three times the arithmetic per shared-memory byte
// for 3//2.  Tiles start at outputs whose p = phi0 + j*D is a multiple of I, so every per-output phase and sample offset
// is a compile-time constant: output o of a thread has phase (o*D) mod I and its window starts (o*D) div I samples after
// the thread's first window.  Same accumulation order as resample_kernel (oldest sample first).
template <int I, int D, int G> struct rs_mp {
    static constexpr int NO = I * G;                          // outputs per thread
    static constexpr int GD = G * D;                          // samples between the windows of neighbouring threads
    static constexpr int OFFMAX = ((NO - 1) * D) / I;         // window offset of the thread's last output
    static constexpr int SK = (GD % 2 == 0) ? 1 : 0;          // skew: odd thread stride in the sample tile (bank conflicts)
    static constexpr int SKO = (NO % 2 == 0) ? 1 : 0;         // same for the output tile
    static constexpr int NTH = 256;
    static constexpr int TILE_OUT = NTH * NO;
    __host__ __device__ static constexpr int xpos(int i) { return i + SK * (i / GD); }
    __host__ __device__ static constexpr int opos(int u) { return u + SKO * (u / NO); }
};

template <typename EX, typename TR, typename EO, int I, int D, int G>
__global__ void __launch_bounds__(256)
resample_mp_kernel(const EX* __restrict__ x, int64_t x_begin, int64_t nx_local, int64_t x_col_stride,
                   const TR* __restrict__ pfb8 /* [I][tpp8] */, int tpp, int tpp8, int64_t n0, int64_t phi0,
                   EO* __restrict__ out, int64_t j_begin, int64_t nout_local, int64_t out_col_stride, int64_t j_tile0,
                   int xtile_len) {
    using M = rs_mp<I, D, G>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TR* bank = reinterpret_cast<TR*>(smem_raw);                                   // I * tpp8
    EX* xs = reinterpret_cast<EX*>(bank + (size_t)I * tpp8);                      // skewed sample tile
    EO* os = reinterpret_cast<EO*>(xs);                                           // reused for the output tile
    const int tid = threadIdx.x;
    const int64_t col = blockIdx.y;
    const int64_t jt = j_tile0 + (int64_t)blockIdx.x * M::TILE_OUT;               // first output of the tile (may be < j_begin)
    const int64_t qt = (phi0 + jt * D) / I;                                       // exact: tiles start at p = 0 (mod I)
    for (int i = tid; i < I * tpp8; i += M::NTH) bank[i] = pfb8[i];
    // xs[xpos(i)] = sample n0 + qt - (tpp-1) + i  (zero outside the stored range)
    const int64_t gb = n0 + qt - (tpp - 1) - x_begin;
    const EX* xb = x + col * x_col_stride + gb;
    const int64_t lo64 = -gb, hi64 = nx_local - gb;
    const int i_lo = lo64 < 0 ? 0 : (lo64 > xtile_len ? xtile_len : (int)lo64);
    const int i_hi = hi64 < 0 ? 0 : (hi64 > xtile_len ? xtile_len : (int)hi64);
    for (int i = tid; i < xtile_len; i += M::NTH) xs[M::xpos(i)] = (i >= i_lo && i < i_hi) ? xb[i] : rs_zero((EX*)nullptr);
    __syncthreads();

    EO acc[M::NO];
#pragma unroll
    for (int o = 0; o < M::NO; ++o) acc[o] = rs_zero((EO*)nullptr);
    const EX* xt = xs + tid * (M::GD + M::SK);                                    // = xs + xpos(tid * GD)
    for (int r0 = 0; r0 < tpp8; r0 += 8) {
        TR h[I][8];
#pragma unroll
        for (int ph = 0; ph < I; ++ph)
#pragma unroll
            for (int q = 0; q < 8; ++q) h[ph][q] = bank[ph * tpp8 + r0 + q];
        EO xv[M::OFFMAX + 8];
        if constexpr (8 % M::GD == 0) {
            // r0 is a multiple of GD: xpos(tid*GD + r0 + q) = xpos(tid*GD) + xpos(r0) + xpos(q), the last one compile-time
            const EX* xr = xt + M::xpos(r0);
#pragma unroll
            for (int q = 0; q < M::OFFMAX + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xr[M::xpos(q)]);
        } else {
#pragma unroll
            for (int q = 0; q < M::OFFMAX + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xs[M::xpos(tid * M::GD + r0 + q)]);
        }
        const bool full = r0 + 8 <= tpp;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (full || r0 + q < tpp) {                       // the zero padding taps never touch a sample
#pragma unroll
                for (int o = 0; o < M::NO; ++o) acc[o] = rs_fma(h[(o * D) % I][q], xv[(o * D) / I + q], acc[o]);
            }
        }
    }
    __syncthreads();                                                              // sample tile no longer needed
#pragma unroll
    for (int o = 0; o < M::NO; ++o) os[M::opos(tid * M::NO + o)] = acc[o];
    __syncthreads();
    // coalesced copy-out of the outputs that fall into [j_begin, j_begin + nout_local)
    EO* oc = out + col * out_col_stride;
    for (int u = tid; u < M::TILE_OUT; u += M::NTH) {
        const int64_t jl = jt + u - j_begin;
        if (jl >= 0 && jl < nout_local) oc[jl] = os[M::opos(u)];
    }
}

// ---------------------------------------------------------------------------------------------- multi-phase, pipelined
// The same register tile as resample_mp_kernel (same products, same accumulation order: bit-identical results) with the
// three things its ncu capture (profiles/r2i_resample.txt) showed removed:
//   * the taps are a KERNEL PARAMETER (at most 64 per phase, rows zero-padded): after unrolling every tap is a constant-bank
//     operand of its FMA -- no tap loads at all (the shared-memory bank cost 24 uniform LDS per 8-tap chunk);
//   * persistent CTAs with a DOUBLE-BUFFERED sample tile: the next tile's samples are fetched with cp.async (LDGSTS, into
//     the same skewed layout) while the current tile is computed, so the global-load latency that stalled the tile's
//     shared-memory stores (long-scoreboard, 20 % of the samples) is off the critical path;
//   * two CTA-wide barriers per tile instead of three, no per-tile tap staging.
// Edge tiles (samples outside the stored range are zero) are filled synchronously with the bounds test.
// The rs_v3 instances also remove what the ncu capture of that version (profiles/r2j_resample.txt: FFMA 54 % of the
// executed instructions although a chunk is 79 % FFMA) showed outside the chunks --
//   * the tap rows are staged ONCE per persistent CTA in shared memory and read with 128-bit broadcast loads (6 per chunk
//     for 3 phases instead of 24 uniform constant loads), which also lets the chunk loop stay ROLLED: two copies of the chunk
//     body (unchecked, and the checked one for the last chunk's padding taps) instead of eight with a uniform branch per tap
//     (97 KB of code);
//   * interior tiles are copied out without the 64-bit bounds tests; single-column launches skip the 64-bit division per tile.
// Same products in the same order as the constant-bank taps: bit-identical.
// Staged tap rows are worth it where the thread's live state (sample window + accumulators + one column group of taps)
// still fits the 80-register budget of three resident CTAs and the window addresses are compile-time offsets (8 % GD == 0);
// the other instances keep the constant-bank taps (they spilled 80-140 bytes with staged rows).
template <typename EO, typename TR, int I, int D, int G> struct rs_v3 {
    using M = rs_mp<I, D, G>;
    static constexpr int est = (M::OFFMAX + 8 + M::NO) * (int)(sizeof(EO) / 4) + I * 4;
    static constexpr bool value = est <= 80 && (8 % M::GD == 0);
};
template <typename TR, int I> struct alignas(16) RsTaps { TR h[I][64]; };

template <typename EX, typename TR, typename EO, int I, int D, int G>
__global__ void __launch_bounds__(256, 3)
resample_mp2_kernel(const EX* __restrict__ x, int64_t x_begin, int64_t nx_local, int64_t x_col_stride,
                    const RsTaps<TR, I> taps, int tpp, int nch, int64_t n0, int64_t phi0,
                    EO* __restrict__ out, int64_t j_begin, int64_t nout_local, int64_t out_col_stride, int64_t j_tile0,
                    int xtile_len, int xbuf_elems, int64_t tiles_per_col, int64_t total_work, const TR* __restrict__ pfb8) {
    using M = rs_mp<I, D, G>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int tid = threadIdx.x;
    constexpr bool V3 = rs_v3<EO, TR, I, D, G>::value;
    TR* hs = reinterpret_cast<TR*>(smem_raw);                                     // rs_v3: [I][64] tap rows, staged once per (persistent) CTA
    EX* xs0 = reinterpret_cast<EX*>(hs + (V3 ? I * 64 : 0));                      // two skewed sample tiles
    if constexpr (V3) {
        for (int i = tid; i < I * 64; i += M::NTH) {
            const int ph = i >> 6, r = i & 63;
            hs[i] = r < nch * 8 ? pfb8[ph * (nch * 8) + r] : TR(0);
        }
    }
    const bool onecol = tiles_per_col >= total_work;                              // no 64-bit division per tile
    EX* xs1 = xs0 + xbuf_elems;
    EO* os = reinterpret_cast<EO*>(xs1 + xbuf_elems);                             // output tile

    // xs[xpos(i)] = sample n0 + qt - (tpp-1) + i of column col (zero outside the stored range), tile `w` of the work list
    auto load_tile = [&](EX* xs, int64_t w) {
        const int64_t col = onecol ? 0 : w / tiles_per_col, tile = w - col * tiles_per_col;
        const int64_t jt = j_tile0 + tile * M::TILE_OUT;                          // first output of the tile (may be < j_begin)
        const int64_t qt = (phi0 + jt * D) / I;                                   // exact: tiles start at p = 0 (mod I)
        const int64_t gb = n0 + qt - (tpp - 1) - x_begin;
        const EX* xb = x + col * x_col_stride + gb;
        if (gb >= 0 && gb + xtile_len <= nx_local) {
            for (int i = tid; i < xtile_len; i += M::NTH) __pipeline_memcpy_async(&xs[M::xpos(i)], &xb[i], sizeof(EX));
        } else {
            const int64_t lo64 = -gb, hi64 = nx_local - gb;
            const int i_lo = lo64 < 0 ? 0 : (lo64 > xtile_len ? xtile_len : (int)lo64);
            const int i_hi = hi64 < 0 ? 0 : (hi64 > xtile_len ? xtile_len : (int)hi64);
            for (int i = tid; i < xtile_len; i += M::NTH) xs[M::xpos(i)] = (i >= i_lo && i < i_hi) ? xb[i] : rs_zero((EX*)nullptr);
        }
    };

    int64_t w = blockIdx.x;
    if (w < total_work) load_tile(xs0, w);
    __pipeline_commit();
    for (int buf = 0; w < total_work; w += gridDim.x, buf ^= 1) {
        const int64_t wn = w + gridDim.x;
        if (wn < total_work) load_tile(buf ? xs0 : xs1, wn);                       // free since the previous tile's second barrier
        __pipeline_commit();
        __pipeline_wait_prior(1);                                                 // this thread's copies of tile w have landed
        __syncthreads();                                                          // ... everybody's; os is free again
        const EX* xs = buf ? xs1 : xs0;

        EO acc[M::NO];
#pragma unroll
        for (int o = 0; o < M::NO; ++o) acc[o] = rs_zero((EO*)nullptr);
        const EX* xt = xs + tid * (M::GD + M::SK);                                // = xs + xpos(tid * GD)
        if constexpr (V3) {
        // one 8-tap chunk: the sample window and the I x 8 taps (128-bit loads) in registers, then I G x 8 multiply-adds.
        // Only the last chunk can hold padding taps (rows are zero-padded to a multiple of 8): it runs the checked copy.
        auto chunk = [&](int c, auto checked) {
            const int r0 = c * 8;
            EO xv[M::OFFMAX + 8];
            if constexpr (8 % M::GD == 0) {
                const EX* xr = xt + M::xpos(r0);
#pragma unroll
                for (int q = 0; q < M::OFFMAX + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xr[M::xpos(q)]);
            } else {
#pragma unroll
                for (int q = 0; q < M::OFFMAX + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xs[M::xpos(tid * M::GD + r0 + q)]);
            }
            constexpr int QV = 16 / (int)sizeof(TR);               // taps per 128-bit load: the taps live in registers QV columns at a time
#pragma unroll
            for (int q0 = 0; q0 < 8; q0 += QV) {
                TR hq[I][QV];
#pragma unroll
                for (int ph = 0; ph < I; ++ph)
                    *reinterpret_cast<uint4*>(&hq[ph][0]) = *reinterpret_cast<const uint4*>(&hs[ph * 64 + r0 + q0]);
#pragma unroll
                for (int qq = 0; qq < QV; ++qq) {
                    const int q = q0 + qq;
                    if (!decltype(checked)::value || r0 + q < tpp) {   // the zero padding taps never touch a sample
#pragma unroll
                        for (int o = 0; o < M::NO; ++o) acc[o] = rs_fma(hq[(o * D) % I][qq], xv[(o * D) / I + q], acc[o]);
                    }
                }
            }
        };
        const int nfull = tpp >> 3;
#pragma unroll 1
        for (int c = 0; c < nfull; ++c) chunk(c, std::false_type());
        if (nfull < nch) chunk(nfull, std::true_type());
        } else {
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            if (c < nch) {
                const int r0 = c * 8;
                EO xv[M::OFFMAX + 8];
                if constexpr (8 % M::GD == 0) {
                    const EX* xr = xt + M::xpos(r0);
#pragma unroll
                    for (int q = 0; q < M::OFFMAX + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xr[M::xpos(q)]);
                } else {
#pragma unroll
                    for (int q = 0; q < M::OFFMAX + 8; ++q) xv[q] = rs_cvt<EO, EX>::get(xs[M::xpos(tid * M::GD + r0 + q)]);
                }
                TR hq[I][8];                                  // the chunk's taps: 128-bit uniform loads from the parameter bank
#pragma unroll
                for (int ph = 0; ph < I; ++ph)
#pragma unroll
                    for (int v = 0; v < 8; v += 16 / (int)sizeof(TR))
                        *reinterpret_cast<uint4*>(&hq[ph][v]) = *reinterpret_cast<const uint4*>(&taps.h[ph][c * 8 + v]);
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    if (r0 + q < tpp) {                       // the zero padding taps never touch a sample
#pragma unroll
                        for (int o = 0; o < M::NO; ++o) acc[o] = rs_fma(hq[(o * D) % I][q], xv[(o * D) / I + q], acc[o]);
                    }
                }
            }
        }
        }
#pragma unroll
        for (int o = 0; o < M::NO; ++o) os[M::opos(tid * M::NO + o)] = acc[o];
        __syncthreads();                                                          // output tile complete; sample tile `buf` free
        // coalesced copy-out of the outputs that fall into [j_begin, j_begin + nout_local)
        const int64_t col = onecol ? 0 : w / tiles_per_col, tile = w - col * tiles_per_col;
        const int64_t jt = j_tile0 + tile * M::TILE_OUT;
        EO* oc = out + col * out_col_stride;
        if (jt >= j_begin && jt + M::TILE_OUT <= j_begin + nout_local) {          // interior tile: no bounds test, 32-bit indices
            EO* ot = oc + (jt - j_begin);
#pragma unroll
            for (int k = 0; k < M::NO; ++k) {
                const int u = tid + k * M::NTH;
                ot[u] = os[M::opos(u)];
            }
        } else
        for (int u = tid; u < M::TILE_OUT; u += M::NTH) {
            const int64_t jl = jt + u - j_begin;
            if (jl >= 0 && jl < nout_local) oc[jl] = os[M::opos(u)];
        }
    }
    __pipeline_wait_prior(0);
}

// ---------------------------------------------------------------------------------------------- arbitrary rate
// filt!(buffer, ::FIRFilter{FIRArbitrary}, x), src/Filters/stream_filt.jl:567-625.  The reference advances a Float64
// phase accumulator serially (acc += delta; carry whole multiples of Nphi into xIdx); output j of a call therefore sits
// at total phase P_j = acc0 + j*delta.  P_j is evaluated here per output in double-double (exact product j*delta, one
// rounding in the final reduction), i.e. to ~1e-15 phases: closer to exact arithmetic than the reference's own running
// sum, whose rounding errors random-walk (~sqrt(j)*Nphi*eps); the interpolated output is continuous in P, so the two
// agree to that order.  Newest input index n_j = n0 + floor(P_j / Nphi), phase phi_j = floor(P_j mod Nphi), alpha_j its
// fraction;  y_j = muladd(dot(dpfb[:, phi], window), alpha, dot(pfb[:, phi], window))  (:606-616), dots oldest sample
// first in the promoted eltype, the final muladd in Float64 as in the reference (alpha is a Float64).
template <typename TR> __device__ __forceinline__ TR arb_mix(TR yu, TR yl, double alpha) { return (TR)fma((double)yu, alpha, (double)yl); }
template <typename TR> __device__ __forceinline__ cx<TR> arb_mix(cx<TR> yu, cx<TR> yl, double alpha) {
    return mkc<TR>((TR)fma((double)yu.x, alpha, (double)yl.x), (TR)fma((double)yu.y, alpha, (double)yl.y));
}

template <typename EX, typename TR, typename EO>
__global__ void __launch_bounds__(RS_NT)
resample_arb_kernel(const EX* __restrict__ x, int64_t nx, const TR* __restrict__ pfb, const TR* __restrict__ dpfb, int tpp,
                    int nphases, int64_t n0, double acc0, double delta, EO* __restrict__ out, int64_t nout, int in_smem) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    TR* ps = reinterpret_cast<TR*>(smem_raw);
    TR* ds = ps + (size_t)nphases * tpp;
    if (in_smem) {
        const int tot = nphases * tpp;
        for (int i = threadIdx.x; i < tot; i += RS_NT) { ps[i] = pfb[i]; ds[i] = dpfb[i]; }
        __syncthreads();
    }
    const int64_t j = (int64_t)blockIdx.x * RS_NT + threadIdx.x;
    if (j >= nout) return;
    const double N = (double)nphases, jd = (double)j;
    const double hi = jd * delta, lo = fma(jd, delta, -hi);          // j*delta = hi + lo exactly
    double q = floor((hi + acc0) / N);
    double r = fma(-q, N, hi);                                       // exact: q*N is an integer, |hi - q*N| small
    r = (r + lo) + acc0;
    while (r < 0.0) { r += N; q -= 1.0; }
    while (r >= N) { r -= N; q += 1.0; }
    const double fl = floor(r);
    const int phi = (int)fl;
    const double alpha = r - fl;
    const int64_t first = n0 + (int64_t)q - (tpp - 1);               // oldest sample of the window
    const TR* hrow = (in_smem ? ps : pfb) + (size_t)phi * tpp;
    const TR* drow = (in_smem ? ds : dpfb) + (size_t)phi * tpp;
    EO yl = rs_zero((EO*)nullptr), yu = rs_zero((EO*)nullptr);
    if (first >= 0 && first + tpp <= nx) {
        const EX* xp = x + first;
        for (int t = 0; t < tpp; ++t) {
            const EO xv = rs_cvt<EO, EX>::get(xp[t]);
            yl = rs_fma(hrow[t], xv, yl);
            yu = rs_fma(drow[t], xv, yu);
        }
    } else {
        for (int t = 0; t < tpp; ++t) {
            const int64_t i = first + t;
            if (i >= 0 && i < nx) {
                const EO xv = rs_cvt<EO, EX>::get(x[i]);
                yl = rs_fma(hrow[t], xv, yl);
                yu = rs_fma(drow[t], xv, yu);
            }
        }
    }
    out[j] = arb_mix(yu, yl, alpha);
}

struct RsPlanImpl {
    int dtype_x = 0, dtype_h = 0, dtype_out = 0;
    int64_t hlen = 0, interp = 1, decim = 1, tpp = 0;
    int device = 0;
    void* d_pfb = nullptr;   // real TR [interp][tpp]
    void* d_pfb8 = nullptr;  // real TR [interp][tpp8]: rows zero-padded to a multiple of 8 taps (tiled kernel)
    void* d_dpfb = nullptr;  // FIRArbitrary: derivative bank taps2pfb([diff(h); 0], Nphi), same layout as d_pfb
    std::vector<float> h8_32;    // host copies of d_pfb8 (kernel-parameter taps of resample_mp2_kernel)
    std::vector<double> h8_64;
    bool arbitrary = false;
    int64_t tpp8 = 0;
    size_t smem_optin = 0;
    DevBuf in, out;
    cudaStream_t stream = nullptr;
};

struct RsArgs {
    const void* x; int64_t x_begin, nx_local, x_col_stride;
    void* out; int64_t j_begin, nout_local, out_col_stride;
    int64_t n0, phi0, ncols;
};

template <typename EX, typename TR, typename EO, int D, int G>
static int rs_launch_tiled(RsPlanImpl* p, const RsArgs& a, cudaStream_t st, bool* done) {
    *done = false;
    const int interp = (int)p->interp;
    int mt = 256 / interp;
    if (mt < 1) return DSPB200_OK;
    const int nthreads = ((interp * mt + 31) / 32) * 32;
    const int tile_out = interp * G * mt;
    // inputs spanned by one tile (+ tap-chunk slack) ; outputs reuse the same region
    const int64_t span = ((int64_t)(tile_out - 1) * D) / interp + p->tpp8 + (G - 1) * D + 16;
    const size_t xbytes = (size_t)(span + 2) * sizeof(EX);
    const size_t region = xbytes > (size_t)tile_out * sizeof(EO) ? xbytes : (size_t)tile_out * sizeof(EO);
    const size_t smem = (size_t)(interp * p->tpp8) * sizeof(TR) + region + 16;
    if (smem > p->smem_optin || smem > 160 * 1024) return DSPB200_OK;
    const int64_t tiles = cdiv(a.nout_local, tile_out);
    if (tiles < 1 || a.ncols < 1) { *done = true; return DSPB200_OK; }
    if (a.ncols > 65535) return DSPB200_OK;                        // gridDim.y limit: generic kernel instead
    DSP_REQUIRE(tiles < (int64_t)0x7fffffff, "too many tiles for one launch");
    auto kern = resample_tiled_kernel<EX, TR, EO, D, G>;
    if (smem > 48 * 1024) DSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<dim3((unsigned)tiles, (unsigned)a.ncols), nthreads, smem, st>>>(
        (const EX*)a.x, a.x_begin, a.nx_local, a.x_col_stride, (const TR*)p->d_pfb8, (int)p->tpp, (int)p->tpp8, interp, mt,
        a.n0, a.phi0, (EO*)a.out, a.j_begin, a.nout_local, a.out_col_stride, (int)span);
    DSP_LAUNCH_OK();
    *done = true;
    return DSPB200_OK;
}

template <typename EX, typename TR, typename EO, int I, int D, int G>
static int rs_launch_mp(RsPlanImpl* p, const RsArgs& a, cudaStream_t st, bool* done) {
    using M = rs_mp<I, D, G>;
    *done = false;
    // samples spanned by one tile: last thread's first window + its last output's offset + the padded tap row
    const int xtile_len = (M::NTH - 1) * M::GD + M::OFFMAX + (int)p->tpp8 + 1;
    const size_t xbytes = (size_t)(M::xpos(xtile_len) + 2) * sizeof(EX);
    const size_t obytes = (size_t)(M::opos(M::TILE_OUT) + 2) * sizeof(EO);
    const size_t smem = (size_t)(I * p->tpp8) * sizeof(TR) + (xbytes > obytes ? xbytes : obytes) + 16;
    if (smem > p->smem_optin || smem > 200 * 1024 || p->tpp8 > 512) return DSPB200_OK;
    if (a.nout_local < 1 || a.ncols < 1) { *done = true; return DSPB200_OK; }
    if (a.ncols > 65535) return DSPB200_OK;
    // tiles are aligned to outputs with p = phi0 + j*D = 0 (mod I): jA = first such j >= 0, grid origin jA - TILE_OUT
    int64_t jA = 0;
    while (((a.phi0 + jA * D) % I) != 0) ++jA;
    const int64_t base = jA - M::TILE_OUT;
    const int64_t k0 = (a.j_begin - base) / M::TILE_OUT;
    const int64_t k1 = (a.j_begin + a.nout_local - 1 - base) / M::TILE_OUT;
    const int64_t tiles = k1 - k0 + 1;
    DSP_REQUIRE(tiles < (int64_t)0x7fffffff, "too many tiles for one launch");
    auto kern = resample_mp_kernel<EX, TR, EO, I, D, G>;
    if (smem > 48 * 1024) DSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<dim3((unsigned)tiles, (unsigned)a.ncols), M::NTH, smem, st>>>(
        (const EX*)a.x, a.x_begin, a.nx_local, a.x_col_stride, (const TR*)p->d_pfb8, (int)p->tpp, (int)p->tpp8, a.n0, a.phi0,
        (EO*)a.out, a.j_begin, a.nout_local, a.out_col_stride, base + k0 * M::TILE_OUT, xtile_len);
    DSP_LAUNCH_OK();
    *done = true;
    return DSPB200_OK;
}

template <typename EX, typename TR, typename EO, int I, int D, int G>
static int rs_launch_mp2(RsPlanImpl* p, const RsArgs& a, cudaStream_t st, bool* done) {
    using M = rs_mp<I, D, G>;
    *done = false;
    if (p->tpp8 > 64) return DSPB200_OK;
    const std::vector<TR>& h8 = [&]() -> const std::vector<TR>& {
        if constexpr (sizeof(TR) == 4) return p->h8_32; else return p->h8_64;
    }();
    if ((int64_t)h8.size() != (int64_t)I * p->tpp8) return DSPB200_OK;
    const int xtile_len = (M::NTH - 1) * M::GD + M::OFFMAX + (int)p->tpp8 + 1;
    const int xbuf_elems = (M::xpos(xtile_len) + 2 + 1) & ~1;                     // even: the second tile stays 16-byte aligned
    const size_t obytes = (size_t)(M::opos(M::TILE_OUT) + 2) * sizeof(EO);
    const size_t smem = 2 * (size_t)xbuf_elems * sizeof(EX) + obytes + 16 + (rs_v3<EO, TR, I, D, G>::value ? (size_t)I * 64 * sizeof(TR) : 0);
    if (smem > p->smem_optin || smem > 72 * 1024) return DSPB200_OK;
    if (a.nout_local < 1 || a.ncols < 1) { *done = true; return DSPB200_OK; }
    // tiles are aligned to outputs with p = phi0 + j*D = 0 (mod I): jA = first such j >= 0, grid origin jA - TILE_OUT
    int64_t jA = 0;
    while (((a.phi0 + jA * D) % I) != 0) ++jA;
    const int64_t base = jA - M::TILE_OUT;
    const int64_t k0 = (a.j_begin - base) / M::TILE_OUT;
    const int64_t k1 = (a.j_begin + a.nout_local - 1 - base) / M::TILE_OUT;
    const int64_t tiles = k1 - k0 + 1, total = tiles * a.ncols;
    RsTaps<TR, I> taps;
    memset(&taps, 0, sizeof(taps));
    for (int ph = 0; ph < I; ++ph)
        for (int64_t r = 0; r < p->tpp8; ++r) taps.h[ph][r] = h8[(size_t)(ph * p->tpp8 + r)];
    auto kern = resample_mp2_kernel<EX, TR, EO, I, D, G>;
    static int per_sm = 0;                                                         // per instantiation: resident CTAs per SM
    if (per_sm == 0) {
        DSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024));
        int n = 0;
        DSP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, M::NTH, smem));
        per_sm = n < 1 ? 1 : n;
    }
    int64_t grid = (int64_t)device_sm_count() * per_sm;
    if (grid > total) grid = total;
    kern<<<(unsigned)grid, M::NTH, smem, st>>>(
        (const EX*)a.x, a.x_begin, a.nx_local, a.x_col_stride, taps, (int)p->tpp, (int)(p->tpp8 / 8), a.n0, a.phi0,
        (EO*)a.out, a.j_begin, a.nout_local, a.out_col_stride, base + k0 * M::TILE_OUT, xtile_len, xbuf_elems, tiles, total,
        (const TR*)p->d_pfb8);
    DSP_LAUNCH_OK();
    *done = true;
    return DSPB200_OK;
}

template <typename EX, typename TR, typename EO>
static int rs_launch(RsPlanImpl* p, const RsArgs& a, cudaStream_t st) {
    if (p->interp >= 2 && p->interp <= 4 && p->decim <= 4 && p->d_pfb8 && a.phi0 >= 0) {
        // multi-phase kernel: G = outputs per phase per thread (Float32 arithmetic: 4; Float64: 2 -- register budget)
        bool done = false;
        constexpr int GM = sizeof(TR) == 4 ? 4 : 2;
        const int key = (int)p->interp * 10 + (int)p->decim;
        switch (key) {                                    // pipelined kernel first (taps as kernel parameters, <= 64 per phase)
            case 21: DSP_TRY((rs_launch_mp2<EX, TR, EO, 2, 1, GM>(p, a, st, &done))); break;
            case 23: DSP_TRY((rs_launch_mp2<EX, TR, EO, 2, 3, GM>(p, a, st, &done))); break;
            case 31: DSP_TRY((rs_launch_mp2<EX, TR, EO, 3, 1, GM>(p, a, st, &done))); break;
            case 32: DSP_TRY((rs_launch_mp2<EX, TR, EO, 3, 2, GM>(p, a, st, &done))); break;
            case 34: DSP_TRY((rs_launch_mp2<EX, TR, EO, 3, 4, GM>(p, a, st, &done))); break;
            case 41: DSP_TRY((rs_launch_mp2<EX, TR, EO, 4, 1, GM>(p, a, st, &done))); break;
            case 43: DSP_TRY((rs_launch_mp2<EX, TR, EO, 4, 3, GM>(p, a, st, &done))); break;
            default: break;
        }
        if (done) return DSPB200_OK;
        switch (key) {
            case 21: DSP_TRY((rs_launch_mp<EX, TR, EO, 2, 1, GM>(p, a, st, &done))); break;
            case 23: DSP_TRY((rs_launch_mp<EX, TR, EO, 2, 3, GM>(p, a, st, &done))); break;
            case 31: DSP_TRY((rs_launch_mp<EX, TR, EO, 3, 1, GM>(p, a, st, &done))); break;
            case 32: DSP_TRY((rs_launch_mp<EX, TR, EO, 3, 2, GM>(p, a, st, &done))); break;
            case 34: DSP_TRY((rs_launch_mp<EX, TR, EO, 3, 4, GM>(p, a, st, &done))); break;
            case 41: DSP_TRY((rs_launch_mp<EX, TR, EO, 4, 1, GM>(p, a, st, &done))); break;
            case 43: DSP_TRY((rs_launch_mp<EX, TR, EO, 4, 3, GM>(p, a, st, &done))); break;
            default: break;
        }
        if (done) return DSPB200_OK;
    }
    if (p->interp <= 128 && p->decim <= 4 && p->d_pfb8) {
        bool done = false;
        // G (outputs per thread) is chosen so that neighbouring threads' windows start G*D samples apart with G*D
        // NOT a multiple of the shared-memory bank period (G = 8, D = 2 measured 78 % conflicting wavefronts)
        constexpr bool F = sizeof(TR) == 4;
        switch (p->decim) {
            case 1: DSP_TRY((rs_launch_tiled<EX, TR, EO, 1, (F ? 7 : 3)>(p, a, st, &done))); break;
            case 2: DSP_TRY((rs_launch_tiled<EX, TR, EO, 2, (F ? 7 : 3)>(p, a, st, &done))); break;
            case 3: DSP_TRY((rs_launch_tiled<EX, TR, EO, 3, (F ? 5 : 3)>(p, a, st, &done))); break;
            default: DSP_TRY((rs_launch_tiled<EX, TR, EO, 4, (F ? 4 : 2)>(p, a, st, &done))); break;
        }
        if (done) return DSPB200_OK;
    }
    const int64_t tiles = cdiv(a.nout_local, RS_NT);
    const int64_t blocks = tiles * a.ncols;
    if (blocks < 1) return DSPB200_OK;
    DSP_REQUIRE(blocks < (int64_t)0x7fffffff, "too many tiles for one launch");
    const size_t bank_bytes = (size_t)(p->interp * p->tpp) * sizeof(TR);
    const int in_smem = bank_bytes <= 96 * 1024;
    const size_t smem = in_smem ? bank_bytes : 0;
    auto kern = resample_kernel<EX, TR, EO>;
    if (smem > 48 * 1024) DSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(unsigned)blocks, RS_NT, smem, st>>>((const EX*)a.x, a.x_begin, a.nx_local, a.x_col_stride, (const TR*)p->d_pfb,
                                                (int)p->tpp, p->interp, p->decim, a.n0, a.phi0, (EO*)a.out, a.j_begin,
                                                a.nout_local, a.out_col_stride, tiles, in_smem);
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

static int rs_run(RsPlanImpl* p, const RsArgs& a, cudaStream_t st) {
    const bool o64 = dtype_is_f64(p->dtype_out);
    switch (p->dtype_x) {
        case DSPB200_F32: return o64 ? rs_launch<float, double, double>(p, a, st) : rs_launch<float, float, float>(p, a, st);
        case DSPB200_F64: return rs_launch<double, double, double>(p, a, st);
        case DSPB200_C32: return o64 ? rs_launch<cx<float>, double, cx<double>>(p, a, st) : rs_launch<cx<float>, float, cx<float>>(p, a, st);
        default: return rs_launch<cx<double>, double, cx<double>>(p, a, st);
    }
}

}  // namespace dspb200

using namespace dspb200;

template <typename EX, typename TR, typename EO>
static int rs_arb_launch(RsPlanImpl* p, const void* x, int64_t nx, int64_t n0, double acc0, double delta, void* out, int64_t nout,
                         cudaStream_t st) {
    const size_t bank_bytes = (size_t)(p->interp * p->tpp) * sizeof(TR) * 2;
    const int in_smem = bank_bytes <= 96 * 1024;
    const size_t smem = in_smem ? bank_bytes : 0;
    auto kern = resample_arb_kernel<EX, TR, EO>;
    if (smem > 48 * 1024) DSP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t blocks = cdiv(nout, RS_NT);
    DSP_REQUIRE(blocks < (int64_t)0x7fffffff, "too many outputs for one launch");
    kern<<<(unsigned)blocks, RS_NT, smem, st>>>((const EX*)x, nx, (const TR*)p->d_pfb, (const TR*)p->d_dpfb, (int)p->tpp,
                                                (int)p->interp, n0, acc0, delta, (EO*)out, nout, in_smem);
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

static int rs_arb_run(RsPlanImpl* p, const void* x, int64_t nx, int64_t n0, double acc0, double delta, void* out, int64_t nout,
                      cudaStream_t st) {
    const bool o64 = p->dtype_out == DSPB200_F64 || p->dtype_out == DSPB200_C64;
    switch (p->dtype_x) {
        case DSPB200_F32:
            return o64 ? rs_arb_launch<float, double, double>(p, x, nx, n0, acc0, delta, out, nout, st)
                       : rs_arb_launch<float, float, float>(p, x, nx, n0, acc0, delta, out, nout, st);
        case DSPB200_F64: return rs_arb_launch<double, double, double>(p, x, nx, n0, acc0, delta, out, nout, st);
        case DSPB200_C32:
            return o64 ? rs_arb_launch<cx<float>, double, cx<double>>(p, x, nx, n0, acc0, delta, out, nout, st)
                       : rs_arb_launch<cx<float>, float, cx<float>>(p, x, nx, n0, acc0, delta, out, nout, st);
        default: return rs_arb_launch<cx<double>, double, cx<double>>(p, x, nx, n0, acc0, delta, out, nout, st);
    }
}

struct dspb200_resample_plan {
    RsPlanImpl impl;
};

extern "C" {

int dspb200_resample_plan_create(dspb200_resample_plan** plan, int dtype_x, int dtype_h, const void* h_host,
                                 int64_t hlen, int64_t interp, int64_t decim) {
    DSP_RANGE("dspb200_resample_plan_create");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    *plan = nullptr;
    DSP_REQUIRE(dtype_valid(dtype_x), "invalid dtype_x %d", dtype_x);
    DSP_REQUIRE(dtype_h == DSPB200_F32 || dtype_h == DSPB200_F64, "taps must be Float32 or Float64");
    DSP_REQUIRE(h_host != nullptr && hlen >= 1, "taps must be non-empty");
    DSP_REQUIRE(interp >= 1 && decim >= 1, "interp and decim must be >= 1");
    dspb200_resample_plan* hnd = new (std::nothrow) dspb200_resample_plan();
    DSP_REQUIRE(hnd != nullptr, "out of host memory");
    RsPlanImpl* p = &hnd->impl;
    p->dtype_x = dtype_x; p->dtype_h = dtype_h; p->hlen = hlen; p->interp = interp; p->decim = decim;
    const bool o64 = dtype_is_f64(dtype_x) || dtype_h == DSPB200_F64;            // promote_type, stream_filt.jl:654
    p->dtype_out = dtype_is_cplx(dtype_x) ? (o64 ? DSPB200_C64 : DSPB200_C32) : (o64 ? DSPB200_F64 : DSPB200_F32);
    p->tpp = (hlen + interp - 1) / interp;                                       // taps2pfb :296
    // bank[phi][r] = hp[phi + (tpp-1-r)*interp]  (pfb column phi, rows top to bottom)
    const size_t cnt = (size_t)(interp * p->tpp);
    std::vector<double> bank64(o64 ? cnt : 0);
    std::vector<float> bank32(o64 ? 0 : cnt);
    for (int64_t phi = 0; phi < interp; ++phi)
        for (int64_t r = 0; r < p->tpp; ++r) {
            const int64_t idx = phi + (p->tpp - 1 - r) * interp;
            double v = 0.0;
            if (idx < hlen) v = dtype_h == DSPB200_F64 ? ((const double*)h_host)[idx] : (double)((const float*)h_host)[idx];
            if (o64) bank64[(size_t)(phi * p->tpp + r)] = v; else bank32[(size_t)(phi * p->tpp + r)] = (float)v;
        }
    const size_t bytes = cnt * (o64 ? 8 : 4);
    p->tpp8 = (p->tpp + 7) / 8 * 8;
    const size_t cnt8 = (size_t)(interp * p->tpp8);
    std::vector<double> b8_64(o64 ? cnt8 : 0, 0.0);
    std::vector<float> b8_32(o64 ? 0 : cnt8, 0.0f);
    for (int64_t phi = 0; phi < interp; ++phi)
        for (int64_t r = 0; r < p->tpp; ++r) {
            if (o64) b8_64[(size_t)(phi * p->tpp8 + r)] = bank64[(size_t)(phi * p->tpp + r)];
            else b8_32[(size_t)(phi * p->tpp8 + r)] = bank32[(size_t)(phi * p->tpp + r)];
        }
    cudaError_t e = cudaGetDevice(&p->device);
    int optin = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, p->device);
    p->smem_optin = (size_t)optin;
    if (e == cudaSuccess) e = cudaMalloc(&p->d_pfb, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_pfb, o64 ? (const void*)bank64.data() : (const void*)bank32.data(), bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_pfb8, cnt8 * (o64 ? 8 : 4));
    if (e == cudaSuccess) e = cudaMemcpy(p->d_pfb8, o64 ? (const void*)b8_64.data() : (const void*)b8_32.data(), cnt8 * (o64 ? 8 : 4), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { const int rc = cuda_fail(e, "tap upload", __FILE__, __LINE__); dspb200_resample_plan_destroy(hnd); return rc; }
    p->h8_32 = b8_32;
    p->h8_64 = b8_64;
    *plan = hnd;
    return DSPB200_OK;
}

int dspb200_resample_out_dtype(const dspb200_resample_plan* plan, int* dtype_out) {
    DSP_REQUIRE(plan && dtype_out, "NULL argument");
    *dtype_out = plan->impl.dtype_out;
    return DSPB200_OK;
}

int dspb200_resample_exec_dev(dspb200_resample_plan* plan, const void* x, int64_t nx, int64_t ncols, int64_t n0,
                              int64_t phi0, void* out, int64_t nout, void* stream) {
    DSP_RANGE("dspb200_resample_exec_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nx >= 0 && ncols >= 0 && nout >= 0, "negative size");
    RsPlanImpl* p = &plan->impl;
    DSP_REQUIRE(n0 >= 0 && phi0 >= 0 && phi0 < p->interp, "bad initial phase");
    if (nout == 0 || ncols == 0) return DSPB200_OK;
    DSP_REQUIRE(out != nullptr && (x != nullptr || nx == 0), "NULL argument");
    RsArgs a{x, 0, nx, nx, out, 0, nout, nout, n0, phi0, ncols};
    return rs_run(p, a, (cudaStream_t)stream);
}

int dspb200_resample_exec_range_dev(dspb200_resample_plan* plan, const void* x_local, int64_t x_begin,
                                    int64_t nx_local, int64_t n0, int64_t phi0, void* out_local, int64_t j_begin,
                                    int64_t nout_local, void* stream) {
    DSP_RANGE("dspb200_resample_exec_range_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    RsPlanImpl* p = &plan->impl;
    DSP_REQUIRE(nx_local >= 0 && nout_local >= 0 && j_begin >= 0, "bad range");
    DSP_REQUIRE(n0 >= 0 && phi0 >= 0 && phi0 < p->interp, "bad initial phase");
    if (nout_local == 0) return DSPB200_OK;
    DSP_REQUIRE(out_local != nullptr && (x_local != nullptr || nx_local == 0), "NULL argument");
    RsArgs a{x_local, x_begin, nx_local, 0, out_local, j_begin, nout_local, 0, n0, phi0, 1};
    return rs_run(p, a, (cudaStream_t)stream);
}

int dspb200_resample_exec(dspb200_resample_plan* plan, const void* x, int64_t nx, int64_t ncols, int64_t n0,
                          int64_t phi0, void* out, int64_t nout) {
    DSP_RANGE("dspb200_resample_exec");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nx >= 0 && ncols >= 0 && nout >= 0, "negative size");
    if (nout == 0 || ncols == 0) return DSPB200_OK;
    DSP_REQUIRE(out != nullptr && (x != nullptr || nx == 0), "NULL argument");
    RsPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    if (!p->stream) DSP_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    const size_t in_bytes = (size_t)(nx * ncols) * dtype_size(p->dtype_x);
    const size_t out_bytes = (size_t)(nout * ncols) * dtype_size(p->dtype_out);
    DSP_TRY(p->in.reserve(in_bytes ? in_bytes : 16));
    DSP_TRY(p->out.reserve(out_bytes));
    if (in_bytes) DSP_CUDA(cudaMemcpyAsync(p->in.p, x, in_bytes, cudaMemcpyHostToDevice, p->stream));
    DSP_TRY(dspb200_resample_exec_dev(plan, p->in.p, nx, ncols, n0, phi0, p->out.p, nout, p->stream));
    DSP_CUDA(cudaMemcpyAsync(out, p->out.p, out_bytes, cudaMemcpyDeviceToHost, p->stream));
    DSP_CUDA(cudaStreamSynchronize(p->stream));
    return DSPB200_OK;
}

// FIRArbitrary(h, rate, Nphi), src/Filters/stream_filt.jl:92-134: pfb = taps2pfb(h, Nphi), dpfb = taps2pfb([diff(h); 0], Nphi)
int dspb200_resample_arb_plan_create(dspb200_resample_plan** plan, int dtype_x, int dtype_h, const void* h_host, int64_t hlen,
                                     int64_t nphases) {
    DSP_RANGE("dspb200_resample_arb_plan_create");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    *plan = nullptr;
    DSP_REQUIRE(dtype_h == DSPB200_F32 || dtype_h == DSPB200_F64, "taps must be Float32 or Float64");
    DSP_REQUIRE(h_host != nullptr && hlen >= 1 && nphases >= 1, "taps must be non-empty and Nphi >= 1");
    DSP_TRY(dspb200_resample_plan_create(plan, dtype_x, dtype_h, h_host, hlen, nphases, 1));
    RsPlanImpl* p = &(*plan)->impl;
    p->arbitrary = true;
    const bool o64 = p->dtype_out == DSPB200_F64 || p->dtype_out == DSPB200_C64;
    const size_t cnt = (size_t)(nphases * p->tpp);
    std::vector<double> bank64(o64 ? cnt : 0);
    std::vector<float> bank32(o64 ? 0 : cnt);
    for (int64_t phi = 0; phi < nphases; ++phi)
        for (int64_t r = 0; r < p->tpp; ++r) {
            const int64_t idx = phi + (p->tpp - 1 - r) * nphases;
            double v = 0.0;                                          // dh = [diff(h); 0] in the taps' own precision
            if (idx + 1 < hlen) {
                if (dtype_h == DSPB200_F64) v = ((const double*)h_host)[idx + 1] - ((const double*)h_host)[idx];
                else v = (double)(float)(((const float*)h_host)[idx + 1] - ((const float*)h_host)[idx]);
            }
            if (o64) bank64[(size_t)(phi * p->tpp + r)] = v; else bank32[(size_t)(phi * p->tpp + r)] = (float)v;
        }
    const size_t bytes = cnt * (o64 ? 8 : 4);
    cudaError_t e = cudaMalloc(&p->d_dpfb, bytes);
    if (e == cudaSuccess) e = cudaMemcpy(p->d_dpfb, o64 ? (const void*)bank64.data() : (const void*)bank32.data(), bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { const int rc = cuda_fail(e, "derivative tap upload", __FILE__, __LINE__); dspb200_resample_plan_destroy(*plan); *plan = nullptr; return rc; }
    return DSPB200_OK;
}

int dspb200_resample_arb_exec_dev(dspb200_resample_plan* plan, const void* x, int64_t nx, int64_t n0, double acc0, double delta,
                                  void* out, int64_t nout, void* stream) {
    DSP_RANGE("dspb200_resample_arb_exec_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    RsPlanImpl* p = &plan->impl;
    DSP_REQUIRE(p->arbitrary, "not an arbitrary-rate plan");
    DSP_REQUIRE(nx >= 0 && nout >= 0, "negative size");
    DSP_REQUIRE(delta > 0.0 && acc0 >= 0.0 && acc0 < (double)p->interp, "bad phase state");
    if (nout == 0) return DSPB200_OK;
    DSP_REQUIRE(out != nullptr && (x != nullptr || nx == 0), "NULL argument");
    return rs_arb_run(p, x, nx, n0, acc0, delta, out, nout, (cudaStream_t)stream);
}

int dspb200_resample_arb_exec(dspb200_resample_plan* plan, const void* x, int64_t nx, int64_t n0, double acc0, double delta,
                              void* out, int64_t nout) {
    DSP_RANGE("dspb200_resample_arb_exec");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nx >= 0 && nout >= 0, "negative size");
    if (nout == 0) return DSPB200_OK;
    DSP_REQUIRE(out != nullptr && (x != nullptr || nx == 0), "NULL argument");
    RsPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    if (!p->stream) DSP_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    const size_t in_bytes = (size_t)nx * dtype_size(p->dtype_x), out_bytes = (size_t)nout * dtype_size(p->dtype_out);
    DSP_TRY(p->in.reserve(in_bytes ? in_bytes : 16));
    DSP_TRY(p->out.reserve(out_bytes));
    if (in_bytes) DSP_CUDA(cudaMemcpyAsync(p->in.p, x, in_bytes, cudaMemcpyHostToDevice, p->stream));
    DSP_TRY(dspb200_resample_arb_exec_dev(plan, p->in.p, nx, n0, acc0, delta, p->out.p, nout, p->stream));
    DSP_CUDA(cudaMemcpyAsync(out, p->out.p, out_bytes, cudaMemcpyDeviceToHost, p->stream));
    DSP_CUDA(cudaStreamSynchronize(p->stream));
    return DSPB200_OK;
}

int dspb200_resample_plan_destroy(dspb200_resample_plan* plan) {
    if (!plan) return DSPB200_OK;
    RsPlanImpl* p = &plan->impl;
    if (p->d_pfb) cudaFree(p->d_pfb);
    if (p->d_pfb8) cudaFree(p->d_pfb8);
    if (p->d_dpfb) cudaFree(p->d_dpfb);
    p->in.release(); p->out.release();
    if (p->stream) cudaStreamDestroy(p->stream);
    delete plan;
    return DSPB200_OK;
}

}  // extern "C"
