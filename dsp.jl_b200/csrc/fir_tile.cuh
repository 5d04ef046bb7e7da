// dspb200 -- register-tiled time-domain FIR (the body of fir_tile_kernel, fir.cu), host-emulable.
//
// filt(b, 1, x) as the reference evaluates it (src/dspbase.jl:95-105, 118-141): one fused multiply-add per tap, oldest tap
// first.  A thread owns G consecutive outputs and walks the taps eight at a time: the 8 taps of a chunk come from 128-bit
// broadcast loads, the G + 7 samples those G x 8 products touch are two 8-sample runs in registers; a chunk loads ONE new
// run (128-bit loads) and the two runs swap roles from chunk to chunk (the loop is unrolled by two: no register shifting).
// So a Float32 chunk is 4 shared-memory loads + the loop counter for 64 multiply-adds -- the one-tap-per-iteration kernel
// it replaced spent two loads and a register shift per 4 multiply-adds and ran at a quarter of the FP32 peak (profiles/r2i_fir.txt).
// The FMA chain of every output is unchanged: bit-identical results.
//
// Taps are padded at the OLD end to a multiple of eight; the padding taps are skipped, never multiplied (0 * Inf = NaN):
// they all sit in the first chunk of the first round, which runs a checked copy of the chunk body.
//
// Shared-memory layout: 16 bytes of padding after every run of 8 elements.  pos(j + 8) = pos(j) + 8 + PADE for every j, so
// a thread's run pointer advances by a constant per chunk (immediate offsets, no per-load address arithmetic), and the
// eight lanes of a 128-bit load phase (thread stride G elements) fall on eight different 16-byte bank groups:
//   4-byte elements, G = 8: lane stride 48 B  -> 0 48 96 16 64 112 32 80 (mod 128);
//   8-byte elements, G = 8: lane stride 80 B  -> 0 80 32 112 64 16 96 48;
//   16-byte elements, G = 4: lane stride 64 B + 16 B per two lanes -> 0 64 16 80 32 96 48 112 (elements 4..7 of a run:
//   64 16 80 32 96 48 112 64, one two-way conflict per phase -- ComplexF64 is bound by the FP64 pipe, not by these loads).
// (tests/host/fir_tile_host_check.cu runs this body for every "thread" on the host against the literal chain.)
#pragma once
#include "common.cuh"
#if !defined(__CUDACC__)
#include <cmath>
#endif

namespace dspb200 {

template <typename T> __host__ __device__ __forceinline__ T fir_fma(T x, T b, T acc) { return fma(x, b, acc); }
// Base.muladd(z::Complex, w::Complex, x::Complex) (base/complex.jl)
template <typename T> __host__ __device__ __forceinline__ cx<T> fir_fma(cx<T> z, cx<T> w, cx<T> x) {
    return mkc<T>(fma(z.x, w.x, -fma(z.y, w.y, -x.x)), fma(z.x, w.y, fma(z.y, w.x, x.y)));
}
template <typename T> __host__ __device__ __forceinline__ T fir_zero(T*) { return T(0); }
template <typename T> __host__ __device__ __forceinline__ cx<T> fir_zero(cx<T>*) { return mkc<T>(T(0), T(0)); }

template <typename E, int NT_> struct fir_geom {
    static constexpr int NT = NT_;
    static constexpr int VEC = 16 / (int)sizeof(E);                    // elements per 128-bit load
    static constexpr int PADE = VEC;                                   // padding elements (16 bytes) after every run of 8
    static constexpr int GS = 8 + PADE;                                // run stride
    static constexpr int G = sizeof(E) == 16 ? 4 : 8;                  // outputs per thread
    static constexpr int TILE = NT * G;                                // outputs per CTA
    static constexpr int KC = 512;                                     // taps per staging round (a multiple of 16)
    __host__ __device__ static constexpr int pos(int j) { return j + PADE * (j >> 3); }
    static constexpr int XS = pos(TILE + KC + 16) + PADE;              // staged samples: TILE + kc + 8 per round
};

// 128-bit move between 16-byte aligned locations (one LDS.128 / register quad on the device)
__host__ __device__ __forceinline__ void fir_copy16(void* dst, const void* src) {
#ifdef __CUDA_ARCH__
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(src);
#else
    memcpy(dst, src, 16);                                               // (the host compiler's strict aliasing rules)
#endif
}

// run of 8 elements: elements 0..3 from lo, 4..7 from hi (the same pointer unless the run straddles a padding gap)
template <typename E> __host__ __device__ __forceinline__ void fir_ld_run(E (&dst)[8], const E* lo, const E* hi) {
    constexpr int VEC = 16 / (int)sizeof(E);
#pragma unroll
    for (int v = 0; v < 8; v += VEC)
        fir_copy16(&dst[v], (v < 4 ? lo : hi) + v);
}

// one chunk: taps t[0..7] (oldest first) against the window lo[0..7] | hi[0..7]; output o, tap q <-> window element o + q
template <typename E, int G, bool CHECKED>
__host__ __device__ __forceinline__ void fir_chunk(E (&acc)[G], const E (&lo)[8], const E (&hi)[8], const E* __restrict__ taps, int nreal_from) {
    E t[8];
    constexpr int VEC = 16 / (int)sizeof(E);
#pragma unroll
    for (int v = 0; v < 8; v += VEC) fir_copy16(&t[v], taps + v);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        if (CHECKED && q < nreal_from) continue;                        // padding tap: skipped, not multiplied
#pragma unroll
        for (int o = 0; o < G; ++o) acc[o] = fir_fma(o + q < 8 ? lo[(o + q) & 7] : hi[(o + q) & 7], t[q], acc[o]);
    }
}

// Staging of one round: samples base .. base + cnt - 1 of the column (zero outside [0, nx)) and the round's taps, oldest first.
template <typename E, int NT>
__host__ __device__ __forceinline__ void fir_stage(int tid, E* xs, E* bs, const E* __restrict__ xc, int64_t nx, int64_t base, int cnt,
                                                   const E* __restrict__ b, int nb, int k_hi, int kc) {
    using Gm = fir_geom<E, NT>;
    for (int j = tid; j < cnt; j += NT) {
        const int64_t g = base + j;
        xs[Gm::pos(j)] = (g >= 0 && g < nx) ? xc[g] : fir_zero((E*)nullptr);
    }
    for (int j = tid; j < kc; j += NT) bs[j] = (k_hi - j < nb) ? b[k_hi - j] : fir_zero((E*)nullptr);
}

// The multiply-adds of one round for thread tid: padded taps k_hi, k_hi - 1, .., k_hi - kc + 1 (kc a multiple of 8),
// xs[pos(j)] = sample (tile start - k_hi + j).  Output o of the thread, padded tap k_hi - c - q <-> xs[G tid + o + c + q].
template <typename E, int NT>
__host__ __device__ __forceinline__ void fir_round(int tid, E (&acc)[fir_geom<E, NT>::G], const E* xs, const E* bs, int nb, int k_hi, int kc) {
    using Gm = fir_geom<E, NT>;
    constexpr int G = Gm::G, GS = Gm::GS;
    const int j0 = G * tid;
    const E* pl = xs + Gm::pos(j0);                  // elements 0..3 of the run that starts at j0 (+ 8 k: + k GS)
    const E* ph = xs + Gm::pos(j0 + 4) - 4;          // elements 4..7
    const E* pt = bs;
    E wa[8], wb[8];
    fir_ld_run<E>(wa, pl, ph);
    pl += GS; ph += GS;
    int c = 0;
    if (k_hi >= nb) {                                // the chunk with the padding taps k_hi .. nb (first chunk of the first round only)
        fir_ld_run<E>(wb, pl, ph);
        fir_chunk<E, G, true>(acc, wa, wb, pt, k_hi - nb + 1);
#pragma unroll
        for (int v = 0; v < 8; ++v) wa[v] = wb[v];
        pl += GS; ph += GS; pt += 8; c = 8;
    }
    for (; c + 16 <= kc; c += 16) {
        fir_ld_run<E>(wb, pl, ph);
        fir_chunk<E, G, false>(acc, wa, wb, pt, 0);
        fir_ld_run<E>(wa, pl + GS, ph + GS);
        fir_chunk<E, G, false>(acc, wb, wa, pt + 8, 0);
        pl += 2 * GS; ph += 2 * GS; pt += 16;
    }
    if (c < kc) {
        fir_ld_run<E>(wb, pl, ph);
        fir_chunk<E, G, false>(acc, wa, wb, pt, 0);
    }
}

}  // namespace dspb200
