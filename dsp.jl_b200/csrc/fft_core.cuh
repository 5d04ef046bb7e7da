// dspb200 -- block-cooperative power-of-two FFT out of shared memory (sm_100a).
//
// Decimation-in-time, FMA form.  N = 16 * 16^k * RL (k = 0..2 twiddled radix-16 passes in shared memory, last radix
// RL in {2, 4, 8, 16}):
//   first pass  plain 16-point DFTs of the residue classes x[c + (N/16) m] straight from the loader (global memory /
//               TMA staging), written as 16 contiguous slots at block rho(c) (mixed-radix digit reversal of c), so
//               that every later pass finds sub-transform r of its group at sub-block r;
//   middle      radix-16 passes at strides 16 and 256, in place (a butterfly reads and writes the same 16 slots);
//   last pass   radix RL at stride N/RL; it leaves X[t + r N/16], r = 0..15, NATURAL order, in the registers of thread
//               t for the consumer (|X|^2 accumulate, x H, store).
// Every radix-R butterfly is a network of radix-2 DIT butterflies  a' = a + w b,  a'' = 2a - a'  -- six FMAs, no
// separate twiddle multiplication: a twiddled radix-16 butterfly costs 192 FP32 instructions and 8 tabulated
// twiddles, six of them tabulated (round 1's DIF form: 168 for the butterfly + 60 for the 15 twiddle products + 36 to
// derive 9 of the 15 twiddles = 264), the plain one 148 (168).
// The inverse is computed with the swap identity IDFT(x) = swap(DFT(swap(x))): only the forward transform exists.
// Overlap-save runs   first | middle | [last, x H, swap, first] | middle | last   with the bracket fused in registers
// (fft_last_pass -> multiply -> fft_bfly16_plain -> fft_store_block).
#pragma once
#include "common.cuh"
#include <math.h>

namespace dspb200 {

// ---------------------------------------------------------------------------------------------- layout
// Padded slot address  p + K (p >> 4) + C8 (p >> 8) + C12 (p >> 12).  K pad elements per 16 slots keep the strided
// passes (lanes = consecutive t inside one 16-slot run) conflict free and every 16-slot run 16-byte aligned, so the
// contiguous first-pass stores move 128 bits at a time (Float32: K = 2; Float64 elements are 16 bytes: K = 1).
// C8 / C12 are chosen per N so that the scattered first-pass stores -- lanes c .. c+7 of a quarter warp write the runs
// rho(c), whose leading digits differ -- fall on eight different 16-byte bank groups (exhaustive search,
// tests/host/fft_core_host_check.cu audits every size: one wavefront per quarter warp).
template <typename T> struct fft_pad { static constexpr int K = sizeof(T) == 4 ? 2 : 1; };
template <typename T> __host__ __device__ constexpr int fft_pad256(int n) {
    if (sizeof(T) == 4) return n == 512 ? 8 : (n == 1024 ? 4 : (n == 8192 ? 4 : 2));
    return n == 512 ? 4 : (n == 1024 ? 2 : (n == 8192 ? 2 : 1));
}
template <typename T> __host__ __device__ constexpr int fft_pad4096(int n) {
    if (sizeof(T) == 4) return n == 8192 ? 2 : (n == 16384 ? 4 : 0);
    return n == 8192 ? 1 : 0;
}
template <typename T, int N> __host__ __device__ __forceinline__ constexpr int padaddr(int p) {
    return p + fft_pad<T>::K * (p >> 4) + fft_pad256<T>(N) * (p >> 8) + fft_pad4096<T>(N) * (p >> 12);
}
template <typename T> __host__ __device__ constexpr int padded_len(int n) {
    // last slot + 1, rounded up to a multiple of 4 so that what follows stays 16-byte aligned
    return ((n - 1) + fft_pad<T>::K * ((n - 1) >> 4) + fft_pad256<T>(n) * ((n - 1) >> 8) + fft_pad4096<T>(n) * ((n - 1) >> 12) + 1 + 3) & ~3;
}
// padded distance of a slot stride S (multiple of 16, or 1): padaddr(base + r S) = padaddr(base) + r padded_stride(S)
// whenever base < S keeps its own bits (base + r S never carries)
template <typename T, int N> __host__ __device__ constexpr int padded_stride(int S) {
    return S + fft_pad<T>::K * (S >> 4) + fft_pad256<T>(N) * (S >> 8) + fft_pad4096<T>(N) * (S >> 12);
}

// two adjacent complex values (16-byte aligned for Float32) in one shared-memory access
template <typename T> __host__ __device__ __forceinline__ void lds2(const cx<T>* p, cx<T>& a, cx<T>& b) {
#ifdef __CUDA_ARCH__
    if constexpr (sizeof(T) == 4) {
        const float4 v = *reinterpret_cast<const float4*>(p);
        a = mkc<T>(v.x, v.y); b = mkc<T>(v.z, v.w);
        return;
    }
#endif
    a = p[0]; b = p[1];
}
template <typename T> __host__ __device__ __forceinline__ void sts2(cx<T>* p, cx<T> a, cx<T> b) {
#ifdef __CUDA_ARCH__
    if constexpr (sizeof(T) == 4) {
        *reinterpret_cast<float4*>(p) = make_float4(a.x, a.y, b.x, b.y);
        return;
    }
#endif
    p[0] = a; p[1] = b;
}

// ---------------------------------------------------------------------------------------------- plan
template <int N> struct fft_plan_traits {
    static_assert((N & (N - 1)) == 0 && N >= 32, "N must be a power of two >= 32");
    static constexpr int log2n() { int l = 0; for (int n = N; n > 1; n >>= 1) ++l; return l; }
    static constexpr int LOGN = log2n();
    static constexpr int Q = N / 16;                        // butterflies per radix-16 pass = residue classes of the first pass
    static constexpr int QL = LOGN - 4;                     // bits left after the first pass
    static constexpr int NMID = QL <= 4 ? 0 : (QL <= 8 ? 1 : 2);          // twiddled radix-16 passes in shared memory
    static constexpr int RL = 1 << (QL - 4 * NMID);         // radix of the last pass: 2, 4, 8 or 16
    static constexpr int SL = N / RL;                       // its stride
    static constexpr int TLK = RL == 16 ? 0 : (N == 16384 ? 1 : RL / 2);   // tabulated twiddles per row of the last-pass table
};

// block (run of 16 slots) of residue class c after the first pass: the digits of c, least significant first in the
// order the passes consume them -- last pass first -- become most significant first
template <int N> __host__ __device__ __forceinline__ int fft_block_of(int c) {
    using P = fft_plan_traits<N>;
    int sub = P::Q / P::RL;
    int pos = (c & (P::RL - 1)) * sub;
    int rest = c / P::RL;
#pragma unroll
    for (int i = 0; i < P::NMID; ++i) {
        sub >>= 4;
        pos += (rest & 15) * sub;
        rest >>= 4;
    }
    return pos;
}

// ---------------------------------------------------------------------------------------------- butterflies
template <typename T> struct fft_const;
template <> struct fft_const<float> {
    static constexpr float SQH = 0.70710678118654752440f;  // sqrt(1/2)
    static constexpr float C8 = 0.92387953251128675613f;   // cos(pi/8)
    static constexpr float S8 = 0.38268343236508977173f;   // sin(pi/8)
};
template <> struct fft_const<double> {
    static constexpr double SQH = 0.70710678118654752440;
    static constexpr double C8 = 0.92387953251128675613;
    static constexpr double S8 = 0.38268343236508977173;
};

// cos(2 pi e / 32), e = 1 .. 7 (compile-time e after unrolling)
template <typename T> __host__ __device__ __forceinline__ constexpr T fft_w32_cos(int e) {
    return e == 1 ? T(0.98078528040323044913L) : e == 2 ? T(0.92387953251128675613L) : e == 3 ? T(0.83146961230254523708L)
         : e == 4 ? T(0.70710678118654752440L) : e == 5 ? T(0.55557023301960222474L) : e == 6 ? T(0.38268343236508977173L)
         : T(0.19509032201612826785L);
}
template <typename T> __host__ __device__ __forceinline__ T fma_(T a, T b, T c) {
#ifdef __CUDA_ARCH__
    return fma(a, b, c);
#else
    return std::fma(a, b, c);
#endif
}
// radix-2 DIT butterflies (a, b) -> (a + w b, a - w b)
template <typename T> __host__ __device__ __forceinline__ void bf_one(cx<T>& a, cx<T>& b) {          // w = 1
    const cx<T> t = a; a = t + b; b = t - b;
}
template <typename T> __host__ __device__ __forceinline__ void bf_mi(cx<T>& a, cx<T>& b) {           // w = -i
    const cx<T> t = a, u = b;
    a = mkc<T>(t.x + u.y, t.y - u.x);
    b = mkc<T>(t.x - u.y, t.y + u.x);
}
// general w = (wr, wi): a' = a + w b in four FMAs, a'' = 2 a - a' in two
template <typename T> __host__ __device__ __forceinline__ void bf_gen(cx<T>& a, cx<T>& b, T wr, T wi) {
    const T px = fma_(wr, b.x, fma_(-wi, b.y, a.x));
    const T py = fma_(wr, b.y, fma_(wi, b.x, a.y));
    b = mkc<T>(fma_(T(2), a.x, -px), fma_(T(2), a.y, -py));
    a = mkc<T>(px, py);
}
// w = -i (wr + i wi) = (wi, -wr)
template <typename T> __host__ __device__ __forceinline__ void bf_gen_mi(cx<T>& a, cx<T>& b, T wr, T wi) { bf_gen<T>(a, b, wi, -wr); }

template <int BITS> __host__ __device__ __forceinline__ constexpr int fft_brev(int p) {
    int r = 0;
    for (int i = 0; i < BITS; ++i) r |= ((p >> i) & 1) << (BITS - 1 - i);
    return r;
}
template <int R> struct fft_log2 { static constexpr int value = R == 2 ? 1 : (R == 4 ? 2 : (R == 8 ? 3 : (R == 16 ? 4 : 5))); };
// tabulated twiddles of one radix-R butterfly: stage k = 1..log2 R holds max(1, 2^(k-2)) values, the rest are -i times one
template <int R> struct fft_tw_count { static constexpr int value = R / 2; };

// Radix-R butterfly, natural order in and out:  v[s] <- sum_r (w^r v[r]) W_R^(r s).
// Stage k (sub-transforms of size 2^k), butterfly m < 2^(k-1) uses omega(k, m) = w^(R / 2^k) W_(2^k)^m; the row `w`
// holds omega(k, m) for k = 1..log2 R, m < max(1, 2^(k-2)) in that order (the second half of a stage is -i times the
// first half: operand permutation).  PLAIN: w = 1, the omegas are constants (1, -i: additions only).
// Stages are template instances so that every loop bound and register index is a compile-time constant.
template <typename T, int R, bool PLAIN, int K> struct fft_bfly_stage {
    static __host__ __device__ __forceinline__ void run(cx<T> (&x)[R], const cx<T>* __restrict__ w) {
        constexpr int half = 1 << (K - 1), quarter = half >> 1;
        constexpr int off = K <= 2 ? K - 1 : (1 << (K - 2));          // row offset of stage K: 0, 1, 2, 4
#pragma unroll
        for (int blk = 0; blk < R; blk += 2 * half) {
#pragma unroll
            for (int m = 0; m < half; ++m) {
                cx<T>& a = x[blk + m];
                cx<T>& b = x[blk + m + half];
                if constexpr (PLAIN) {
                    if (m == 0) bf_one<T>(a, b);
                    else if (m == quarter) bf_mi<T>(a, b);
                    else {
                        // W_(2^K)^mm, mm = m mod quarter in 1 .. quarter-1: K = 3 -> W_8; K = 4 -> W_16^(1,2,3); K = 5 -> W_32^(1..7)
                        const int mm = m < quarter ? m : m - quarter;
                        const int e = mm * (32 >> K);                  // exponent over 32: 1 .. 7
                        const T wr = fft_w32_cos<T>(e), wi = -fft_w32_cos<T>(8 - e);      // sin(2 pi e / 32) = cos(2 pi (8 - e) / 32)
                        if (m < quarter) bf_gen<T>(a, b, wr, wi); else bf_gen_mi<T>(a, b, wr, wi);
                    }
                } else {
                    if (quarter == 0 || m < quarter) { const cx<T> o = w[off + m]; bf_gen<T>(a, b, o.x, o.y); }
                    else { const cx<T> o = w[off + m - quarter]; bf_gen_mi<T>(a, b, o.x, o.y); }
                }
            }
        }
        if constexpr ((1 << K) < R) fft_bfly_stage<T, R, PLAIN, K + 1>::run(x, w);
    }
};
template <typename T, int R, bool PLAIN>
__host__ __device__ __forceinline__ void fft_bfly(cx<T> (&v)[R], const cx<T>* __restrict__ w) {
    constexpr int QB = fft_log2<R>::value;
    cx<T> x[R];
#pragma unroll
    for (int p = 0; p < R; ++p) x[p] = v[fft_brev<QB>(p)];
    fft_bfly_stage<T, R, PLAIN, 1>::run(x, w);
#pragma unroll
    for (int s = 0; s < R; ++s) v[s] = x[s];
}
template <typename T> __host__ __device__ __forceinline__ void fft_bfly16_plain(cx<T> (&v)[16]) {
    fft_bfly<T, 16, true>(v, nullptr);
}

// ---------------------------------------------------------------------------------------------- twiddle tables
// Radix-16 passes at stride S (sub-transforms of size M = 16 S) need w = W_M^t, t < S: one row of 8 values per t, 6 of them stored.
// S is 16 or 256 for every supported N, so two small tables serve all sizes: T16[16][8] (M = 256), T256[256][8]
// (M = 4096); they are staged in shared memory (0.75 KB + 12 KB for Float32).  The last pass, when its radix RL is below
// 16, reads its row (RL/2 values of W_N^t-based omegas, t < N/RL) from a per-plan table TL in global memory
// (L1-resident); for the 16384-point Float32 transform TL holds W_N^t alone (32 KB, staged in shared memory: the CTA is
// alone on its SM anyway) and the second value of the radix-4 row, W_N^2t, is its square.
// stored values per row (of the 8 a butterfly uses): 6, the two products with W8 are formed on the fly -- except for the
// 16384-point transform, whose CTA is alone on its SM anyway and has the room for all 8 (conv kernel: 0.547 -> 0.530 ms)
__host__ __device__ constexpr int fft_tw_row(long long n) { return n == 16384 ? 8 : 6; }
__host__ __device__ constexpr int fft_tw16_len(long long n) { return 16 * fft_tw_row(n); }
__host__ __device__ constexpr int fft_tw256_len(long long n) { return 256 * fft_tw_row(n); }

template <typename T> struct FftCtx {
    cx<T>* sm;                      // padded data buffer, padded_len(N) elements
    const cx<T>* t16;               // shared: T16
    const cx<T>* t256;              // shared: T256
    const cx<T>* tl;                // last-pass table: global, or shared when fft_tl_in_smem
};

template <typename T, int N> __host__ __device__ constexpr bool fft_tl_in_smem() {
    // 16384: W_N^t alone, 32 KB; 512 / 1024 / 2048: the whole last-pass table, 2 / 4 / 8 KB (several CTAs per SM still fit)
    return sizeof(T) == 4 && (N == 16384 || N == 512 || N == 1024 || N == 2048);
}
template <int N> __host__ __device__ constexpr int fft_tl_len() { return (N / fft_plan_traits<N>::RL) * fft_plan_traits<N>::TLK; }
template <int N> __host__ __device__ constexpr bool fft_uses_t16() { return N >= 256; }
template <int N> __host__ __device__ constexpr bool fft_uses_t256() { return N >= 4096; }

// shared-memory footprint of a fused transform of size N (data + twiddle tables), in elements of cx<T>
template <typename T, int N> __host__ __device__ constexpr int fft_smem_elems() {
    return padded_len<T>(N) + (fft_uses_t16<N>() ? fft_tw16_len(N) : 0) + (fft_uses_t256<N>() ? fft_tw256_len(N) : 0) +
           (fft_tl_in_smem<T, N>() ? fft_tl_len<N>() : 0);
}

template <typename T> __host__ __device__ __forceinline__ cx<T> ldtw(const cx<T>* __restrict__ tw, int j) {
#ifndef __CUDA_ARCH__
    return tw[j];
#else
    if constexpr (sizeof(T) == 4) {
        float2 v = __ldg(reinterpret_cast<const float2*>(tw) + j);
        return mkc<T>(v.x, v.y);
    } else {
        double2 v = __ldg(reinterpret_cast<const double2*>(tw) + j);
        return mkc<T>(v.x, v.y);
    }
#endif
}

// Table layout in memory: NOT row-major (rows of 64 bytes would put the lanes t, t+1, .. of a quarter warp on only two
// 16-byte bank groups: a 4-way conflict on every twiddle load -- measured: +20 % on the conv kernel).  Float32: pair-major,
// element pair i (values 2i, 2i+1) of row t is the 16-byte word i * S + t -- consecutive lanes read consecutive words;
// Float64: element-major, value i of row t is the 16-byte word i * S + t.
template <typename T> __host__ __device__ __forceinline__ constexpr int fft_tw_index(int i, int t, int S) {
    return sizeof(T) == 4 ? (((i >> 1) * S + t) * 2 + (i & 1)) : (i * S + t);
}
// The 8 twiddles of butterfly t of the radix-16 pass at stride S, in the order fft_bfly wants them
// (w^8, w^4, w^2, W8 w^2, w, W16 w, W8 w, W16^3 w).  Six are stored -- (w^8, w^4), (w^2, w), (W16 w, W16^3 w): three
// 16-byte words for Float32 -- and the two products with W8 = (1 - i)/sqrt(2) cost two additions and two multiplications
// each: a quarter less twiddle traffic and 4 KB less shared memory per CTA than storing all eight (the complex
// 4096-point Welch kernel keeps its window table in shared memory next to two resident CTAs only with the 12 KB table).
template <typename T> __host__ __device__ __forceinline__ cx<T> mul_w8(cx<T> a) {
    const T h = fft_const<T>::SQH;
    return mkc<T>(h * (a.x + a.y), h * (a.y - a.x));
}
template <typename T, int S, int ROW> __host__ __device__ __forceinline__ void load_tw8(const cx<T>* __restrict__ tab, int t, cx<T> (&w)[8]) {
    cx<T> s[ROW];
    if constexpr (sizeof(T) == 4) {
#pragma unroll
        for (int i = 0; i < ROW; i += 2) lds2<T>(tab + fft_tw_index<T>(i, t, S), s[i], s[i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < ROW; ++i) s[i] = tab[fft_tw_index<T>(i, t, S)];
    }
    if constexpr (ROW == 8) {
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = s[i];
    } else {
        w[0] = s[0]; w[1] = s[1]; w[2] = s[2]; w[3] = mul_w8<T>(s[2]);
        w[4] = s[3]; w[5] = s[4]; w[6] = mul_w8<T>(s[3]); w[7] = s[5];
    }
}

// shared-memory elements of the twiddle tables alone (fft_smem_elems minus the data buffer)
template <typename T, int N> __host__ __device__ constexpr int fft_table_elems() { return fft_smem_elems<T, N>() - padded_len<T>(N); }

// Copy the twiddle tables a transform of size N needs from global memory into shared memory at `tabs` (fft_table_elems
// elements) and return the context for the data buffer `data`.  Must be followed by a barrier over all NT staging
// threads before the first pass that uses them.
template <typename T, int N, int NT>
__device__ __forceinline__ FftCtx<T> fft_make_ctx_at(cx<T>* data, cx<T>* tabs, const cx<T>* __restrict__ g16,
                                                       const cx<T>* __restrict__ g256, const cx<T>* __restrict__ gtl, int tid) {
    FftCtx<T> c;
    c.sm = data;
    cx<T>* s16 = tabs;
    cx<T>* s256 = s16 + (fft_uses_t16<N>() ? fft_tw16_len(N) : 0);
    c.t16 = s16;
    c.t256 = s256;
    c.tl = gtl;
    if constexpr (fft_uses_t16<N>()) {
        for (int i = tid; i < fft_tw16_len(N); i += NT) s16[i] = g16[i];
    }
    if constexpr (fft_uses_t256<N>()) {
        for (int i = tid; i < fft_tw256_len(N); i += NT) s256[i] = g256[i];
    }
    if constexpr (fft_tl_in_smem<T, N>()) {
        cx<T>* sl = s256 + (fft_uses_t256<N>() ? fft_tw256_len(N) : 0);
        for (int i = tid; i < fft_tl_len<N>(); i += NT) sl[i] = gtl[i];
        c.tl = sl;
    }
    return c;
}
// tables right behind the data buffer (the single-transform kernels)
template <typename T, int N, int NT>
__device__ __forceinline__ FftCtx<T> fft_make_ctx(cx<T>* smem, const cx<T>* __restrict__ g16, const cx<T>* __restrict__ g256,
                                                    const cx<T>* __restrict__ gtl, int tid) {
    return fft_make_ctx_at<T, N, NT>(smem, smem + padded_len<T>(N), g16, g256, gtl, tid);
}

// ---------------------------------------------------------------------------------------------- passes
// Thread -> butterfly map of every pass: b = tid + it * NT, b < N/16.
// Barriers (callers): first pass | full | middle 1 | group | middle 2 | full | last pass.  Between the two middle
// passes only the 256 butterflies of one 4096-point sub-transform exchange data: threads tid / 256 synchronise among
// themselves (named barrier), the groups drift apart and de-phase their load / math / store bursts inside one CTA.
template <int NT> __device__ __forceinline__ void fft_group256_sync(int tid) {
#ifdef __CUDA_ARCH__
    if constexpr (NT <= 256) __syncthreads();
    else asm volatile("bar.sync %0, %1;" ::"r"(1 + (tid >> 8)), "r"(256) : "memory");
#endif
}

// Barrier scope of one transform: the whole CTA, or one of several independent thread groups of a CTA (the multi-group
// Welch kernel runs up to three transforms per CTA that share one copy of the twiddle tables and of the window).
struct FftCtaScope {
    __device__ __forceinline__ void sync() const {
#ifdef __CUDA_ARCH__
        __syncthreads();
#endif
    }
};
template <int NTG> struct FftGroupScope {
    int id;                                          // named barrier 8 + group index (1..4: 256-thread sub-transform groups, 5..7: load gating)
    __device__ __forceinline__ void sync() const {
#ifdef __CUDA_ARCH__
        asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NTG) : "memory");
#endif
    }
};

// Load gating.  After a CTA-wide barrier all 32 warps of a 1024-thread CTA issue their 16-20 shared-memory loads at once;
// the loads of all warps interleave in the memory pipe, every warp gets its operands only when nearly ALL loads have been
// served, and the FMA pipe idles for the whole load phase (ncu: LDS = 6 % of the instructions, 28 % of the stall samples;
// issue slots 56 % busy).  With gating the 256-thread waves take turns: wave k issues its loads only after wave k-1 has
// issued all of its own (named barrier 4+k: wave k-1 arrives, wave k waits), so wave 0 computes while wave 1 loads, ...
// Only used in passes that follow a CTA-wide barrier (a group-synchronised pass is already de-phased, and its waves may
// be a whole pass apart, which would break the arrive/wait pairing).
template <int NT> __device__ __forceinline__ void fft_gate_wait(int tid) {
#ifdef __CUDA_ARCH__
    if constexpr (NT > 256) {
        const int k = tid >> 8;
        if (k > 0) asm volatile("bar.sync %0, 512;" ::"r"(4 + k) : "memory");
    }
#endif
}
template <int NT> __device__ __forceinline__ void fft_gate_open(int tid) {
#ifdef __CUDA_ARCH__
    if constexpr (NT > 256) {
        const int k = tid >> 8;
        if (k < NT / 256 - 1) asm volatile("bar.arrive %0, 512;" ::"r"(5 + k) : "memory");
    }
#endif
}

// store the outputs of a plain first-pass butterfly of residue class cidx: 16 contiguous slots at block rho(cidx)
template <typename T, int N> __host__ __device__ __forceinline__ void fft_store_block(cx<T>* sm, int cidx, const cx<T> (&v)[16]) {
    cx<T>* p = sm + padaddr<T, N>(16 * fft_block_of<N>(cidx));
#pragma unroll
    for (int r = 0; r < 16; r += 2) sts2<T>(p + r, v[r], v[r + 1]);
}

// First pass: ld0(j, it, r) supplies sample j = c + r N/16 of the (natural order) input.  SYNC places one
// __syncthreads() between the first butterfly's arithmetic and its stores (the caller's previous pass still reads the
// buffer): the global loads and the butterfly overlap the other warps' tail of that pass.
template <typename T, int N, int NT, bool SYNC, class Ld0, class Scope = FftCtaScope>
__host__ __device__ __forceinline__ void fft_first_pass(const FftCtx<T>& c, int tid, Ld0 ld0, Scope sc = Scope()) {
    constexpr int Q = fft_plan_traits<N>::Q;
    constexpr int ITERS = (Q + NT - 1) / NT;
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int b = tid + it * NT;
        const bool active = (Q % NT == 0) || b < Q;
        cx<T> v[16];
        if (active) {
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = ld0(b + r * Q, it, r);
            fft_bfly16_plain<T>(v);
        }
#ifdef __CUDA_ARCH__
        if constexpr (SYNC) { if (it == 0) sc.sync(); }
#endif
        if (active) fft_store_block<T, N>(c.sm, b, v);
    }
}

// Twiddled radix-16 pass at stride S (16 or 256), in place.
template <typename T, int N, int NT, int S, bool GATE = false>
__host__ __device__ __forceinline__ void fft_pass16(const FftCtx<T>& c, int tid) {
    static_assert(S == 16 || S == 256, "radix-16 pass with an unsupported stride");
    constexpr int Q = fft_plan_traits<N>::Q;
    constexpr int ITERS = (Q + NT - 1) / NT;
    constexpr int PS = padded_stride<T, N>(S);
    const cx<T>* tab = S == 16 ? c.t16 : c.t256;
    if constexpr (ITERS == 2 && Q % NT == 0) {
        // two butterflies per thread: both are loaded before either is transformed (the compiler cannot move the second
        // one's shared-memory loads above the first one's stores -- it cannot prove the slots distinct)
        const int b0 = tid, b1 = tid + NT;
        const int t0 = b0 & (S - 1), t1 = b1 & (S - 1);
        cx<T>* p0 = c.sm + padaddr<T, N>((b0 / S) * (16 * S) + t0);
        cx<T>* p1 = c.sm + padaddr<T, N>((b1 / S) * (16 * S) + t1);
        cx<T> v0[16], v1[16], w0[8], w1[8];
        if constexpr (GATE) fft_gate_wait<NT>(tid);
        load_tw8<T, S, fft_tw_row(N)>(tab, t0, w0);
#pragma unroll
        for (int r = 0; r < 16; ++r) v0[r] = p0[r * PS];
        load_tw8<T, S, fft_tw_row(N)>(tab, t1, w1);
#pragma unroll
        for (int r = 0; r < 16; ++r) v1[r] = p1[r * PS];
        if constexpr (GATE) fft_gate_open<NT>(tid);
        fft_bfly<T, 16, false>(v0, w0);
#pragma unroll
        for (int r = 0; r < 16; ++r) p0[r * PS] = v0[r];
        fft_bfly<T, 16, false>(v1, w1);
#pragma unroll
        for (int r = 0; r < 16; ++r) p1[r * PS] = v1[r];
        return;
    }
#pragma unroll 1
    for (int it = 0; it < ITERS; ++it) {
        const int b = tid + it * NT;
        if (Q % NT != 0 && b >= Q) break;
        const int t = b & (S - 1);
        cx<T>* p = c.sm + padaddr<T, N>((b / S) * (16 * S) + t);
        cx<T> v[16], w[8];
        if constexpr (GATE && ITERS == 1) fft_gate_wait<NT>(tid);
        load_tw8<T, S, fft_tw_row(N)>(tab, t, w);
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = p[r * PS];
        if constexpr (GATE && ITERS == 1) fft_gate_open<NT>(tid);
        fft_bfly<T, 16, false>(v, w);
#pragma unroll
        for (int r = 0; r < 16; ++r) p[r * PS] = v[r];
    }
}

// The passes between the first and the last one.  Entered after a full barrier (the first pass is complete), leaves
// after a full barrier: the last pass may start.
template <typename T, int N, int NT, class Scope = FftCtaScope>
__device__ __forceinline__ void fft_middle(const FftCtx<T>& c, int tid, Scope sc = Scope()) {
    constexpr int NMID = fft_plan_traits<N>::NMID;
    static_assert(NMID < 2 || std::is_same<Scope, FftCtaScope>::value, "thread groups run transforms of at most 4096 points");
    if constexpr (NMID >= 1) {
        fft_pass16<T, N, NT, 16, true>(c, tid);
        if constexpr (NMID == 2) {
            fft_group256_sync<NT>(tid);
            fft_pass16<T, N, NT, 256>(c, tid);
        }
        sc.sync();
    }
}

// Last pass of thread unit tp = tid + it * NT < N/16: on return v[r] = X[tp + r N/16].
template <typename T, int N, int GATE_NT = 0>
__host__ __device__ __forceinline__ void fft_last_pass(const FftCtx<T>& c, int tp, cx<T> (&v)[16], int tid = 0) {
    using P = fft_plan_traits<N>;
    constexpr int Q = P::Q, RL = P::RL;
    if constexpr (GATE_NT > 256) fft_gate_wait<GATE_NT>(tid);
    {
        // padaddr(tp + r Q) = padaddr(tp) + padaddr(r Q): tp < Q never carries into the bits of r Q (compile-time offsets)
        const cx<T>* p = c.sm + padaddr<T, N>(tp);
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = p[padaddr<T, N>(r * Q)];
    }
    if constexpr (GATE_NT > 256) fft_gate_open<GATE_NT>(tid);
    if constexpr (RL == 16) {
        cx<T> w[8];
        load_tw8<T, Q, fft_tw_row(N)>(Q == 16 ? c.t16 : c.t256, tp, w);
        fft_bfly<T, 16, false>(v, w);
    } else {
        constexpr int NBF = 16 / RL;                 // butterflies of this thread: a = 0 .. NBF-1, t = tp + Q a
        constexpr int TLK = P::TLK;
#pragma unroll
        for (int a = 0; a < NBF; ++a) {
            const int t = tp + Q * a;
            cx<T> w[RL / 2];
            if constexpr (N == 16384) {              // row = (W^2t, W^t), W^2t by squaring
                const cx<T> w1 = fft_tl_in_smem<T, N>() ? c.tl[t] : ldtw<T>(c.tl, t);
                w[1] = w1;
                w[0] = mkc<T>(fma_(w1.x, w1.x, -(w1.y * w1.y)), (w1.x + w1.x) * w1.y);
            } else {
#pragma unroll
                for (int i = 0; i < TLK; ++i) w[i] = fft_tl_in_smem<T, N>() ? c.tl[t * TLK + i] : ldtw<T>(c.tl, t * TLK + i);
            }
            cx<T> u[RL];
#pragma unroll
            for (int j = 0; j < RL; ++j) u[j] = v[a + NBF * j];
            fft_bfly<T, RL, false>(u, w);
#pragma unroll
            for (int j = 0; j < RL; ++j) v[a + NBF * j] = u[j];
        }
    }
}

// The last pass in chunks of one butterfly (a radix below 16 gives a thread 16/RL butterflies): chunk a leaves
// u[j] = X[tp + (a + (16/RL) j) N/16], j < RL.  Lets a consumer that streams its outputs away (global stores) keep only RL
// values live at a time -- the overlap-save kernel holds the next unit's 16 prefetched samples in registers meanwhile.
template <int N> struct fft_last_chunks {
    static constexpr int RL = fft_plan_traits<N>::RL;
    static constexpr int COUNT = 16 / RL;                 // 1 when the last pass is a radix-16 pass
};
template <typename T, int N, int A>
__device__ __forceinline__ void fft_last_pass_chunk(const FftCtx<T>& c, int tp, cx<T> (&u)[fft_plan_traits<N>::RL]) {
    using P = fft_plan_traits<N>;
    constexpr int Q = P::Q, RL = P::RL, NBF = 16 / RL;
    const cx<T>* p = c.sm + padaddr<T, N>(tp);
#pragma unroll
    for (int j = 0; j < RL; ++j) u[j] = p[padaddr<T, N>((A + NBF * j) * Q)];
    if constexpr (RL == 16) {
        cx<T> w[8];
        load_tw8<T, Q, fft_tw_row(N)>(Q == 16 ? c.t16 : c.t256, tp, w);
        fft_bfly<T, 16, false>(u, w);
    } else {
        const int t = tp + Q * A;
        cx<T> w[RL / 2];
        if constexpr (N == 16384) {
            const cx<T> w1 = fft_tl_in_smem<T, N>() ? c.tl[t] : ldtw<T>(c.tl, t);
            w[1] = w1;
            w[0] = mkc<T>(fma_(w1.x, w1.x, -(w1.y * w1.y)), (w1.x + w1.x) * w1.y);
        } else {
#pragma unroll
            for (int i = 0; i < P::TLK; ++i) w[i] = fft_tl_in_smem<T, N>() ? c.tl[t * P::TLK + i] : ldtw<T>(c.tl, t * P::TLK + i);
        }
        fft_bfly<T, RL, false>(u, w);
    }
}

// Whole forward transform: natural order in (ld0), natural order out: stl(k, it, r, X[k]) with k = tp + r N/16 from
// the registers of the last pass.  All threads of the block must call it; contains __syncthreads().
template <typename T, int N, int NT, class Ld0, class StLast>
__device__ __forceinline__ void fft_forward(const FftCtx<T>& c, int tid, Ld0 ld0, StLast stlast) {
    constexpr int Q = fft_plan_traits<N>::Q;
    constexpr int ITERS = (Q + NT - 1) / NT;
    fft_first_pass<T, N, NT, false>(c, tid, ld0);
    __syncthreads();
    fft_middle<T, N, NT>(c, tid);
#pragma unroll
    for (int it = 0; it < ITERS; ++it) {
        const int tp = tid + it * NT;
        if (Q % NT != 0 && tp >= Q) break;
        cx<T> v[16];
        fft_last_pass<T, N>(c, tp, v);
#pragma unroll
        for (int r = 0; r < 16; ++r) stlast(tp + r * Q, it, r, v[r]);
    }
}

// ---------------------------------------------------------------------------------------------- host side
// omega(k, m) rows for w = exp(-2 pi i * num / den), radix R: long-double trig, rounded once
template <typename T> inline void fft_fill_row(cx<T>* row, int R, long long num, long long den, int limit = 1 << 30) {
    const long double PI2 = 6.283185307179586476925286766559005768L;
    int qb = 0;
    for (int r = R; r > 1; r >>= 1) ++qb;
    int idx = 0;
    for (int k = 1; k <= qb; ++k) {
        const int cnt = k <= 2 ? 1 : (1 << (k - 2));
        for (int m = 0; m < cnt; ++m) {
            // w^(R / 2^k) * W_(2^k)^m
            const long double a = -PI2 * ((long double)num * (long double)(R >> k) / (long double)den + (long double)m / (long double)(1 << k));
            if (idx < limit) row[idx] = mkc<T>((T)cosl(a), (T)sinl(a));
            ++idx;
        }
    }
}
template <typename T> inline void fft_fill_tables(cx<T>* t16, cx<T>* t256, long long n) {
    cx<T> row[8];
    const int nrow = fft_tw_row(n);
    const int keep6[6] = {0, 1, 2, 4, 5, 7};                // w^8, w^4, w^2, w, W16 w, W16^3 w (see load_tw8)
    for (int t = 0; t < 16; ++t) {
        fft_fill_row<T>(row, 16, t, 256);
        for (int i = 0; i < nrow; ++i) t16[fft_tw_index<T>(i, t, 16)] = row[nrow == 8 ? i : keep6[i]];
    }
    for (int t = 0; t < 256; ++t) {
        fft_fill_row<T>(row, 16, t, 4096);
        for (int i = 0; i < nrow; ++i) t256[fft_tw_index<T>(i, t, 256)] = row[nrow == 8 ? i : keep6[i]];
    }
}
// last-pass table of a transform of size n (runtime): rows t < n / RL
inline void fft_last_radix(long long n, int* rl, int* tlk) {
    int logn = 0;
    for (long long m = n; m > 1; m >>= 1) ++logn;
    const int ql = logn - 4;
    const int nmid = ql <= 4 ? 0 : (ql <= 8 ? 1 : 2);
    *rl = 1 << (ql - 4 * nmid);
    *tlk = *rl == 16 ? 0 : (n == 16384 ? 1 : *rl / 2);
}
inline long long fft_tl_len_rt(long long n) {
    int rl, tlk;
    fft_last_radix(n, &rl, &tlk);
    return (n / rl) * tlk;
}
template <typename T> inline void fft_fill_tl(cx<T>* tl, long long n) {
    int rl, tlk;
    fft_last_radix(n, &rl, &tlk);
    if (tlk == 0) return;
    const long double PI2 = 6.283185307179586476925286766559005768L;
    for (long long t = 0; t < n / rl; ++t) {
        if (n == 16384) {
            const long double a = -PI2 * (long double)t / (long double)n;
            tl[t] = mkc<T>((T)cosl(a), (T)sinl(a));
        } else {
            fft_fill_row<T>(tl + t * tlk, rl, t, n);
        }
    }
}

// Threads per block for a fused transform of size N: one radix-16 butterfly per thread up to 256 threads.
template <int N> struct fft_threads {
    static constexpr int NB16 = N / 16;
    static constexpr int value = NB16 < 64 ? 64 : (NB16 > 512 ? 512 : (NB16 > 256 ? 256 : NB16));
};
// __launch_bounds__ min-blocks: cap Float32 kernels at 128 registers (512 resident threads per SM at least);
// Float64 butterflies need the full register file.
template <typename T, int N> struct fft_minblocks {
    static constexpr int value = sizeof(T) == 8 ? 1 : (fft_threads<N>::value >= 512 ? 1 : 512 / fft_threads<N>::value);
};

}  // namespace dspb200
