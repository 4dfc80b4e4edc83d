// b200sd -- library-level plumbing of the C ABI: error text, launch counter, TMA descriptor encode.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>

#include "common.cuh"

static thread_local char g_err[512] = "";
std::atomic<long long> g_b200sd_launches{0};

void b200sd_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* b200sd_last_error(void) { return g_err; }

// The opt-in to > 48 KB of dynamic shared memory is a per-DEVICE attribute of a kernel function: set once per (kernel address,
// device) under a mutex (the C ABI may be called from several threads, and a process may drive several GPUs).
#include <map>
#include <utility>
cudaError_t b200sd_opt_in_smem_impl(const void* kernel, int bytes, bool max_carveout) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, int> configured;      // (kernel, device) -> bytes opted in
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair(kernel, dev);
    auto it = configured.find(key);
    if (it != configured.end() && it->second >= bytes) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return e;
    if (max_carveout) {
        e = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
        if (e != cudaSuccess) return e;
    }
    configured[key] = bytes;
    return cudaSuccess;
}
extern "C" int b200sd_version(void) { return 103; }
extern "C" int64_t b200sd_launch_count(void) { return g_b200sd_launches.load(); }

// ---- in-graph timers: events recorded with cudaEventRecordExternal, so that a captured plan can carry a timestamp between
// any two of its kernels and a replay yields per-kernel times under the REAL conditions of the step (cold weights streaming
// from HBM, the true predecessor in L2) -- what bench.py's roofline uses.
#include <vector>
static std::vector<cudaEvent_t> g_timers;
extern "C" int b200sd_timer_reserve(int n) {
    B200SD_REQUIRE(n >= 0 && n <= (1 << 20), "timer_reserve: bad count %d", n);
    while ((int)g_timers.size() < n) {
        cudaEvent_t e;
        B200SD_CUDA(cudaEventCreate(&e));
        g_timers.push_back(e);
    }
    return B200SD_OK;
}
extern "C" int b200sd_timer_record(int i, b200sd_stream_t stream) {
    B200SD_REQUIRE(i >= 0 && i < (int)g_timers.size(), "timer_record: index %d not reserved", i);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    B200SD_CUDA(cudaStreamIsCapturing(s, &st));
    B200SD_CUDA(cudaEventRecordWithFlags(g_timers[i], s, st == cudaStreamCaptureStatusActive ? cudaEventRecordExternal : cudaEventRecordDefault));
    return B200SD_OK;
}
extern "C" int b200sd_timer_elapsed_ms(int i, int j, float* ms) {
    B200SD_REQUIRE(ms && i >= 0 && j >= 0 && i < (int)g_timers.size() && j < (int)g_timers.size(), "timer_elapsed: bad index");
    B200SD_CUDA(cudaEventElapsedTime(ms, g_timers[i], g_timers[j]));
    return B200SD_OK;
}

int b200sd_num_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    }
    return sms;
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static encode_tiled_fn get_encode_fn() {
    static encode_tiled_fn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<encode_tiled_fn>(p);
    });
    return fn;
}

int b200sd_make_tmap(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapSwizzle swizzle,
                     CUtensorMapDataType dtype) {
    encode_tiled_fn fn = get_encode_fn();
    B200SD_REQUIRE(fn != nullptr, "cuTensorMapEncodeTiled driver entry point unavailable");
    cuuint64_t gdim[5];
    cuuint64_t gstr[5];
    cuuint32_t bdim[5];
    cuuint32_t estr[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bdim[i] = box[i];
        estr[i] = 1;
        if (i > 0) gstr[i - 1] = strides_bytes[i];
    }
    CUresult r = fn(out, dtype, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bdim, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B200SD_REQUIRE(r == CUDA_SUCCESS,
                   "cuTensorMapEncodeTiled failed (%d): rank %d dims [%llu %llu %llu %llu] box [%u %u %u %u] base %p",
                   (int)r, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                   (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
                   rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0, base);
    return B200SD_OK;
}
