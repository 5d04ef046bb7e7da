// dspb200 -- time-domain FIR: filt(b, 1, x) / tdfilt (src/dspbase.jl:26-66, 95-154; src/Filters/filt.jl:431-443).
//
// The reference runs a transposed direct-form loop whose state update is si[j] = muladd(x_i, b[j+1], si[j+1])
// (:95-105, and the unrolled NTuple form :118-141), which unrolls to
//     y[i] = fma(x[i], b[1], fma(x[i-1], b[2], ... fma(x[i-nb+2], b[nb-1], x[i-nb+1]*b[nb])))
// i.e. one fused multiply-add per tap, oldest tap first.  This kernel evaluates exactly that chain per
// output, so Float32/Float64 results match the reference bit for bit on FMA hardware.
// fir_tile_kernel (fir_tile.cuh) evaluates it: a thread owns 8 consecutive outputs (4 for ComplexF64) and walks the taps 8
// at a time from 128-bit loads, at 62-69 % of the FP32 peak.  The x tile (+ tap-chunk halo) and the tap chunk are staged in
// shared memory, padded so that the sliding-window reads are bank-conflict free.  It replaced a one-tap-per-iteration kernel
// on every measured shape (profiles/README.md, FIR table; measured in round 2 with a variant since removed; see the history
// before this commit).
#include "common.cuh"
#include "fir_tile.cuh"
#include <new>

namespace dspb200 {

// fir_tile.cuh: a thread owns G consecutive outputs, 8 taps per chunk, two 8-sample register runs that swap roles.
template <typename E, int NT>
__global__ void __launch_bounds__(NT)
fir_tile_kernel(const E* __restrict__ x, int64_t nx, int64_t tiles_per_col, const E* __restrict__ b, int nb,
                E* __restrict__ out) {
    using Gm = fir_geom<E, NT>;
    constexpr int G = Gm::G;
    __shared__ __align__(16) E xs[Gm::XS];
    __shared__ __align__(16) E bs[Gm::KC];
    const int tid = threadIdx.x;
    const int64_t col = blockIdx.x / tiles_per_col;
    const int64_t tile = blockIdx.x % tiles_per_col;
    const int64_t i0 = tile * Gm::TILE;
    const E* xc = x + col * nx;
    E* oc = out + col * nx;
    E acc[G];
#pragma unroll
    for (int o = 0; o < G; ++o) acc[o] = fir_zero((E*)nullptr);
    const int nb8 = (nb + 7) & ~7;                                      // taps nb .. nb8-1 are padding (skipped)
    for (int k_hi = nb8 - 1; k_hi >= 0; k_hi -= Gm::KC) {
        const int kc = k_hi + 1 < Gm::KC ? k_hi + 1 : Gm::KC;           // padded taps k_hi, k_hi-1, .., k_hi-kc+1 (a multiple of 8)
        __syncthreads();
        fir_stage<E, NT>(tid, xs, bs, xc, nx, i0 - k_hi, Gm::TILE + kc + 8, b, nb, k_hi, kc);
        __syncthreads();
        fir_round<E, NT>(tid, acc, xs, bs, nb, k_hi, kc);
    }
    const int64_t i = i0 + (int64_t)G * tid;
    if (i + G <= nx && (reinterpret_cast<uintptr_t>(oc + i) & 15) == 0) {
#pragma unroll
        for (int v = 0; v < G; v += Gm::VEC) *reinterpret_cast<uint4*>(oc + i + v) = *reinterpret_cast<const uint4*>(&acc[v]);
    } else {
#pragma unroll
        for (int o = 0; o < G; ++o)
            if (i + o < nx) oc[i + o] = acc[o];
    }
}

struct FirPlanImpl {
    int dtype = 0;
    int64_t nb = 0;
    int device = 0;
    void* d_b = nullptr;
    DevBuf in, out;
    cudaStream_t stream = nullptr;
};

}  // namespace dspb200

using namespace dspb200;

struct dspb200_fir_plan {
    FirPlanImpl impl;
};

extern "C" {

int dspb200_fir_plan_create(dspb200_fir_plan** plan, int dtype, const void* b_host, int64_t nb) {
    DSP_RANGE("dspb200_fir_plan_create");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    *plan = nullptr;
    DSP_REQUIRE(dtype_valid(dtype), "invalid dtype %d", dtype);
    DSP_REQUIRE(b_host != nullptr && nb >= 1, "filter vector b must be non-empty");   // ArgumentError src/dspbase.jl:28
    DSP_REQUIRE(nb < (int64_t(1) << 30), "filter too long");
    dspb200_fir_plan* h = new (std::nothrow) dspb200_fir_plan();
    DSP_REQUIRE(h != nullptr, "out of host memory");
    FirPlanImpl* p = &h->impl;
    p->dtype = dtype; p->nb = nb;
    cudaError_t e = cudaGetDevice(&p->device);
    if (e == cudaSuccess) e = cudaMalloc(&p->d_b, (size_t)nb * dtype_size(dtype));
    if (e == cudaSuccess) e = cudaMemcpy(p->d_b, b_host, (size_t)nb * dtype_size(dtype), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { const int rc = cuda_fail(e, "tap upload", __FILE__, __LINE__); dspb200_fir_plan_destroy(h); return rc; }
    *plan = h;
    return DSPB200_OK;
}

int dspb200_fir_exec_dev(dspb200_fir_plan* plan, const void* x, int64_t nx, int64_t ncols, void* out, void* stream) {
    DSP_RANGE("dspb200_fir_exec_dev");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nx >= 0 && ncols >= 0, "negative size");
    if (nx == 0 || ncols == 0) return DSPB200_OK;
    DSP_REQUIRE(x && out, "NULL argument");
    FirPlanImpl* p = &plan->impl;
    cudaStream_t st = (cudaStream_t)stream;
#define FIR_TILED(E_) do {                                                                                   \
        /* short inputs: 128-thread tiles, so that the tiles spread evenly over the SMs */                   \
        const bool small = cdiv(nx, fir_geom<E_, 256>::TILE) * ncols < (int64_t)8 * device_sm_count();       \
        const int64_t tiles = cdiv(nx, small ? fir_geom<E_, 128>::TILE : fir_geom<E_, 256>::TILE), blocks = tiles * ncols; \
        DSP_REQUIRE(blocks < (int64_t)0x7fffffff, "too many tiles for one launch");                          \
        if (small) fir_tile_kernel<E_, 128><<<(unsigned)blocks, 128, 0, st>>>((const E_*)x, nx, tiles, (const E_*)p->d_b, (int)p->nb, (E_*)out); \
        else fir_tile_kernel<E_, 256><<<(unsigned)blocks, 256, 0, st>>>((const E_*)x, nx, tiles, (const E_*)p->d_b, (int)p->nb, (E_*)out); \
    } while (0)
    switch (p->dtype) {
        case DSPB200_F32: FIR_TILED(float); break;
        case DSPB200_F64: FIR_TILED(double); break;
        case DSPB200_C32: FIR_TILED(cx<float>); break;
        default: FIR_TILED(cx<double>); break;
    }
#undef FIR_TILED
    DSP_LAUNCH_OK();
    return DSPB200_OK;
}

int dspb200_fir_exec(dspb200_fir_plan* plan, const void* x, int64_t nx, int64_t ncols, void* out) {
    DSP_RANGE("dspb200_fir_exec");
    DSP_REQUIRE(plan != nullptr, "plan is NULL");
    DSP_REQUIRE(nx >= 0 && ncols >= 0, "negative size");
    if (nx == 0 || ncols == 0) return DSPB200_OK;
    DSP_REQUIRE(x && out, "NULL argument");
    FirPlanImpl* p = &plan->impl;
    DSP_CUDA(cudaSetDevice(p->device));
    if (!p->stream) DSP_CUDA(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    const size_t bytes = (size_t)(nx * ncols) * dtype_size(p->dtype);
    DSP_TRY(p->in.reserve(bytes));
    DSP_TRY(p->out.reserve(bytes));
    DSP_CUDA(cudaMemcpyAsync(p->in.p, x, bytes, cudaMemcpyHostToDevice, p->stream));
    DSP_TRY(dspb200_fir_exec_dev(plan, p->in.p, nx, ncols, p->out.p, p->stream));
    DSP_CUDA(cudaMemcpyAsync(out, p->out.p, bytes, cudaMemcpyDeviceToHost, p->stream));
    DSP_CUDA(cudaStreamSynchronize(p->stream));
    return DSPB200_OK;
}

int dspb200_fir_plan_destroy(dspb200_fir_plan* plan) {
    if (!plan) return DSPB200_OK;
    FirPlanImpl* p = &plan->impl;
    if (p->d_b) cudaFree(p->d_b);
    p->in.release(); p->out.release();
    if (p->stream) cudaStreamDestroy(p->stream);
    delete plan;
    return DSPB200_OK;
}

}  // extern "C"
