// dspb200 -- runtime entry points: errors, device selection, memory helpers.
#include "common.cuh"
#include <atomic>
#include <cufft.h>
#include <mutex>
#include <vector>

namespace dspb200 {

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char* what, const char* file, int line) {
    set_error("CUDA error %d (%s) in %s at %s:%d", (int)e, cudaGetErrorString(e), what, file, line);
    cudaGetLastError();
    return e == cudaErrorMemoryAllocation ? DSPB200_ENOMEM : DSPB200_ECUDA;
}

int device_sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
    return n;
}

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

// ---- plan cache / scratch arena of the plan-less entry points
static std::recursive_mutex g_conv_mutex;
ConvenienceLock::ConvenienceLock() { g_conv_mutex.lock(); }
ConvenienceLock::~ConvenienceLock() { g_conv_mutex.unlock(); }

struct PlanEntry {
    int device, rank, type;
    long long n[3], idist, odist, batch;
    bool embed;
    cufftHandle handle;
    uint64_t stamp;
};
static std::vector<PlanEntry> g_plans;
static uint64_t g_plan_clock = 0;

int plan_cache_get(int* handle, int rank, const long long* n, bool embed, long long idist, long long odist, int type, long long batch) {
    int dev = 0;
    DSP_CUDA(cudaGetDevice(&dev));
    long long nn[3] = {1, 1, 1};
    for (int d = 0; d < rank; ++d) nn[d] = n[d];
    for (auto& e : g_plans) {
        if (e.device == dev && e.rank == rank && e.type == type && e.embed == embed && e.idist == idist && e.odist == odist &&
            e.batch == batch && e.n[0] == nn[0] && e.n[1] == nn[1] && e.n[2] == nn[2]) {
            e.stamp = ++g_plan_clock;
            *handle = (int)e.handle;
            return DSPB200_OK;
        }
    }
    cufftHandle h = 0;
    size_t ws = 0;
    cufftResult r = cufftCreate(&h);
    if (r == CUFFT_SUCCESS)
        r = cufftMakePlanMany64(h, rank, nn, embed ? nn : nullptr, 1, embed ? idist : 0, embed ? nn : nullptr, 1, embed ? odist : 0,
                                (cufftType)type, batch, &ws);
    if (r != CUFFT_SUCCESS) {
        if (h) cufftDestroy(h);
        set_error("cuFFT error %d creating a cached plan", (int)r);
        return DSPB200_ECUFFT;
    }
    if (g_plans.size() >= 32) {                       // evict the least recently used plan
        size_t lru = 0;
        for (size_t i = 1; i < g_plans.size(); ++i) if (g_plans[i].stamp < g_plans[lru].stamp) lru = i;
        cufftDestroy(g_plans[lru].handle);
        g_plans.erase(g_plans.begin() + (long)lru);
    }
    g_plans.push_back(PlanEntry{dev, rank, type, {nn[0], nn[1], nn[2]}, idist, odist, batch, embed, h, ++g_plan_clock});
    *handle = (int)h;
    return DSPB200_OK;
}

static DevBuf g_scratch[8];
DevBuf& scratch_buf(int slot) { return g_scratch[slot & 7]; }
void scratch_trim(size_t keep_bytes) {
    for (auto& b : g_scratch) if (b.cap > keep_bytes) b.release();
}

}  // namespace dspb200

using namespace dspb200;

extern "C" {

int dspb200_version(void) { return DSPB200_VERSION; }
const char* dspb200_last_error(void) { return g_err; }
int64_t dspb200_launch_count(void) { return g_launches.load(); }

int dspb200_device_count(int* count) {
    DSP_REQUIRE(count != nullptr, "count is NULL");
    *count = 0;
    DSP_CUDA(cudaGetDeviceCount(count));
    return DSPB200_OK;
}

int dspb200_set_device(int device) {
    DSP_CUDA(cudaSetDevice(device));
    return DSPB200_OK;
}

int dspb200_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem, size_t* l2_bytes) {
    int dev = 0;
    DSP_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    DSP_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    if (total_mem) *total_mem = p.totalGlobalMem;
    if (l2_bytes) *l2_bytes = (size_t)p.l2CacheSize;
    return DSPB200_OK;
}

int dspb200_malloc(void** dptr, size_t bytes) {
    DSP_REQUIRE(dptr != nullptr, "dptr is NULL");
    *dptr = nullptr;
    if (bytes == 0) return DSPB200_OK;
    DSP_CUDA(cudaMalloc(dptr, bytes));
    return DSPB200_OK;
}
int dspb200_free(void* dptr) {
    if (dptr) DSP_CUDA(cudaFree(dptr));
    return DSPB200_OK;
}
int dspb200_host_alloc(void** hptr, size_t bytes) {
    DSP_REQUIRE(hptr != nullptr, "hptr is NULL");
    *hptr = nullptr;
    if (bytes == 0) return DSPB200_OK;
    DSP_CUDA(cudaHostAlloc(hptr, bytes, cudaHostAllocDefault));
    return DSPB200_OK;
}
int dspb200_host_free(void* hptr) {
    if (hptr) DSP_CUDA(cudaFreeHost(hptr));
    return DSPB200_OK;
}
int dspb200_memcpy_h2d(void* dst, const void* src, size_t bytes, void* stream) {
    if (bytes == 0) return DSPB200_OK;
    DSP_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return DSPB200_OK;
}
int dspb200_memcpy_d2h(void* dst, const void* src, size_t bytes, void* stream) {
    if (bytes == 0) return DSPB200_OK;
    DSP_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return DSPB200_OK;
}
int dspb200_stream_sync(void* stream) {
    DSP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return DSPB200_OK;
}

}  // extern "C"
