// dspb200 -- the 16384-point transform as 32 x 32 x 16 (one shared-memory middle pass per transform instead of two).
//
// Same decimation-in-time FMA-form butterflies and the same conventions as fft_core.cuh -- natural order in, natural order
// out, swap identity for the inverse -- with radix-32 butterflies (64 data registers, 512 threads, one butterfly per thread):
//   first pass   plain 32-point DFTs of the residue classes x[c + 512 m], written as 32 contiguous slots at block rho(c);
//   middle pass  radix 32 at stride 32 (sub-transforms of 1024 points), in place, twiddles W_1024^t from T32[32][16];
//   last pass    radix 16 at stride 1024, twiddles W_16384^t from T1024[1024][8]; thread t leaves X[t + 1024 r], r < 16.
// Timing probes on the 16 x 16 x 16 x 4 kernel (profiles/README.md) put 42 % of its time in the four LSU-bound middle
// passes; this plan has two per overlap-save block.  Shared memory: data 145 KB + T32 4 KB + T1024 64 KB = 213 KB.
#pragma once
#include "fft_core.cuh"

namespace dspb200 {
namespace r32 {

constexpr int N = 16384;
constexpr int NT = 512;                 // threads: one radix-32 butterfly each, two radix-16 butterflies in the last pass
constexpr int Q32 = N / 32;             // 512 residue classes / radix-32 butterflies per pass
constexpr int Q16 = N / 16;             // 1024 butterflies of the last pass
constexpr int T32_LEN = 32 * 16;        // stored twiddles of the middle pass (all 16 of a radix-32 butterfly)
constexpr int T1024_LEN = 1024 * 8;

// padded slot address: the usual 2 per 16 and 2 per 256, plus 2 per 1024 -- the scattered first-pass stores of a quarter
// warp go to blocks 1024 slots apart (rho(c) = 32 (c mod 16) + c / 16) and must fall on eight different 16-byte bank groups
__host__ __device__ __forceinline__ constexpr int pad(int p) { return p + 2 * (p >> 4) + 2 * (p >> 8) + 2 * (p >> 10); }
__host__ __device__ constexpr int padded_len() { return (pad(N - 1) + 1 + 3) & ~3; }
__host__ __device__ __forceinline__ constexpr int block_of(int c) { return (c & 15) * 32 + (c >> 4); }
template <typename T> __host__ __device__ constexpr int smem_elems() { return padded_len() + T32_LEN + T1024_LEN; }

template <typename T> struct Ctx {
    cx<T>* sm;
    const cx<T>* t32;       // shared: pair-major, word i*32 + t holds values 2i, 2i+1 of row t
    const cx<T>* t1024;     // shared: pair-major, word i*1024 + t
};

template <typename T>
__device__ __forceinline__ Ctx<T> make_ctx(cx<T>* smem, const cx<T>* __restrict__ g32, const cx<T>* __restrict__ g1024, int tid) {
    Ctx<T> c;
    c.sm = smem;
    cx<T>* s32 = smem + padded_len();
    cx<T>* s1024 = s32 + T32_LEN;
    for (int i = tid; i < T32_LEN; i += NT) s32[i] = g32[i];
    for (int i = tid; i < T1024_LEN; i += NT) s1024[i] = g1024[i];
    c.t32 = s32;
    c.t1024 = s1024;
    return c;
}

// plain 32-point butterfly of residue class c on registers, then 32 contiguous slots at block rho(c)
template <typename T> __host__ __device__ __forceinline__ void store_block(cx<T>* sm, int c, const cx<T> (&v)[32]) {
    cx<T>* p = sm + pad(32 * block_of(c));
#pragma unroll
    for (int r = 0; r < 32; r += 2) sts2<T>(p + pad(r), v[r], v[r + 1]);
}

// middle pass: radix 32 at stride 32, butterfly b = (blk, t): slots blk*1024 + t + 32 r
template <typename T> __host__ __device__ __forceinline__ void middle_pass(const Ctx<T>& c, int tid) {
    const int t = tid & 31;
    cx<T>* p = c.sm + pad((tid >> 5) * 1024 + t);
    cx<T> v[32], w[16];
#pragma unroll
    for (int i = 0; i < 16; i += 2) lds2<T>(c.t32 + ((i >> 1) * 32 + t) * 2, w[i], w[i + 1]);
#pragma unroll
    for (int r = 0; r < 32; ++r) v[r] = p[pad(32 * r)];
    fft_bfly<T, 32, false>(v, w);
#pragma unroll
    for (int r = 0; r < 32; ++r) p[pad(32 * r)] = v[r];
}

// last pass of thread unit tp < 1024: v[r] = X[tp + 1024 r]
template <typename T> __host__ __device__ __forceinline__ void last_pass(const Ctx<T>& c, int tp, cx<T> (&v)[16]) {
    const cx<T>* p = c.sm + pad(tp);
    cx<T> w[8];
#pragma unroll
    for (int i = 0; i < 8; i += 2) lds2<T>(c.t1024 + ((i >> 1) * 1024 + tp) * 2, w[i], w[i + 1]);
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = p[pad(1024 * r)];
    fft_bfly<T, 16, false>(v, w);
}

// host side: the two tables
template <typename T> inline void fill_tables(cx<T>* t32, cx<T>* t1024) {
    cx<T> row[16];
    for (int t = 0; t < 32; ++t) {
        fft_fill_row<T>(row, 32, t, 1024);
        for (int i = 0; i < 16; ++i) t32[((i >> 1) * 32 + t) * 2 + (i & 1)] = row[i];
    }
    for (int t = 0; t < 1024; ++t) {
        fft_fill_row<T>(row, 16, t, 16384);
        for (int i = 0; i < 8; ++i) t1024[((i >> 1) * 1024 + t) * 2 + (i & 1)] = row[i];
    }
}

}  // namespace r32
}  // namespace dspb200
