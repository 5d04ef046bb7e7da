// dspb200 -- common device/host helpers (complex type, dtype traits, error plumbing).
#pragma once
#include <cuda_runtime.h>
#include <nvtx3/nvToolsExt.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdarg.h>
#include <type_traits>

#include "../../include/dspb200.h"

namespace dspb200 {

// ----------------------------------------------------------------------------------------------
// Interleaved complex (layout-identical to Julia's Complex{T}, float2 / double2).
template <typename T>
struct alignas(2 * sizeof(T)) cx {
    T x, y;
};

template <typename T> __host__ __device__ __forceinline__ cx<T> mkc(T a, T b) { cx<T> r; r.x = a; r.y = b; return r; }
template <typename T> __host__ __device__ __forceinline__ cx<T> operator+(cx<T> a, cx<T> b) { return mkc<T>(a.x + b.x, a.y + b.y); }
template <typename T> __host__ __device__ __forceinline__ cx<T> operator-(cx<T> a, cx<T> b) { return mkc<T>(a.x - b.x, a.y - b.y); }
template <typename T> __host__ __device__ __forceinline__ cx<T> cmul(cx<T> a, cx<T> b) {
    return mkc<T>(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
template <typename T> __host__ __device__ __forceinline__ cx<T> cscale(cx<T> a, T s) { return mkc<T>(a.x * s, a.y * s); }
template <typename T> __host__ __device__ __forceinline__ cx<T> cconj(cx<T> a) { return mkc<T>(a.x, -a.y); }
template <typename T> __host__ __device__ __forceinline__ cx<T> cswap(cx<T> a) { return mkc<T>(a.y, a.x); }
// multiply by -i
template <typename T> __host__ __device__ __forceinline__ cx<T> mul_mi(cx<T> a) { return mkc<T>(a.y, -a.x); }
template <typename T> __host__ __device__ __forceinline__ T cabs2(cx<T> a) { return a.x * a.x + a.y * a.y; }

// ----------------------------------------------------------------------------------------------
// dtype traits
template <typename E> struct elt_traits;
template <> struct elt_traits<float>       { using real = float;  static constexpr bool is_cplx = false; };
template <> struct elt_traits<double>      { using real = double; static constexpr bool is_cplx = false; };
template <> struct elt_traits<cx<float>>   { using real = float;  static constexpr bool is_cplx = true; };
template <> struct elt_traits<cx<double>>  { using real = double; static constexpr bool is_cplx = true; };

inline size_t dtype_size(int dt) {
    switch (dt) {
        case DSPB200_F32: return 4;
        case DSPB200_F64: return 8;
        case DSPB200_C32: return 8;
        case DSPB200_C64: return 16;
    }
    return 0;
}
inline bool dtype_is_cplx(int dt) { return dt == DSPB200_C32 || dt == DSPB200_C64; }
inline bool dtype_is_f64(int dt) { return dt == DSPB200_F64 || dt == DSPB200_C64; }
inline bool dtype_valid(int dt) { return dt >= 0 && dt <= 3; }

// ----------------------------------------------------------------------------------------------
// error plumbing (thread-local message; the C ABI never throws)
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define DSP_CUDA(call)                                                              \
    do {                                                                            \
        cudaError_t e__ = (call);                                                   \
        if (e__ != cudaSuccess) return ::dspb200::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)

#define DSP_REQUIRE(cond, ...)                    \
    do {                                          \
        if (!(cond)) {                            \
            ::dspb200::set_error(__VA_ARGS__);    \
            return DSPB200_EINVALID;              \
        }                                         \
    } while (0)

// NVTX range around every C-ABI entry point that does device work (SURVEY.md section 5: the reference has no tracing; this
// is what makes the library's calls visible on an Nsight timeline).  Header-only NVTX3: a no-op unless a tool is attached.
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
};
#define DSP_RANGE(name) ::dspb200::NvtxRange nvtx_range__(name)

#define DSP_TRY(expr)               \
    do {                            \
        int rc__ = (expr);          \
        if (rc__ != DSPB200_OK) return rc__; \
    } while (0)

// Device scratch buffer that only grows (owned by plans).
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return DSPB200_OK;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e)); cudaGetLastError(); return DSPB200_ENOMEM; }
        cap = bytes;
        return DSPB200_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

int device_sm_count();
void count_launch(int n = 1);

// cuFFT plans and device scratch of the plan-less convenience entry points (conv_fft, conv_nd, hilbert, periodogram2) are
// cached: round 1 created and destroyed two plans and up to six allocations per call.  `plan_cache_get` returns a handle
// owned by the cache (never destroy it); `embed` selects inembed = onembed = n with the given distances (hilbert's
// real -> complex plan), otherwise the default packed layout.  The cache keeps the 32 most recently used plans per
// process; callers serialise on `convenience_lock()` for the duration of the call (the entry points are synchronous).
int plan_cache_get(int* handle, int rank, const long long* n, bool embed, long long idist, long long odist, int type, long long batch);
DevBuf& scratch_buf(int slot);            // per-process grow-only device buffers, slot 0..7
void scratch_trim(size_t keep_bytes);     // release the buffers larger than keep_bytes
struct ConvenienceLock { ConvenienceLock(); ~ConvenienceLock(); };

// after every kernel launch
#define DSP_LAUNCH_OK()                                                              \
    do {                                                                            \
        ::dspb200::count_launch(1);                                                 \
        cudaError_t e__ = cudaGetLastError();                                       \
        if (e__ != cudaSuccess) return ::dspb200::cuda_fail(e__, "kernel launch", __FILE__, __LINE__); \
    } while (0)
static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Programmatic dependent launch (sm_90+).  The persistent kernels of a pipeline (overlap-save -> Welch -> finalize -> next
// overlap-save) are launched with programmatic stream serialisation: a kernel's CTAs may become resident as soon as the
// previous kernel's CTAs leave an SM, stage their twiddle tables / window (constants since plan creation) and then block
// in `pdl_wait()` until the previous grid has completed and its memory is visible -- the launch gap and the table prologue
// (68 KB per CTA for the 16384-point kernel) overlap the previous kernel's tail instead of following it.  EVERY thread
// executes pdl_wait() before its first access to anything a preceding kernel could have written or still be reading, so
// the chain is transitive.  Without the launch attribute both instructions are no-ops.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KA, typename... A>
static inline cudaError_t launch_pdl(void (*kern)(KA...), unsigned grid, unsigned block, size_t smem, cudaStream_t st, A... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, KA(args)...);
}
#endif

}  // namespace dspb200
