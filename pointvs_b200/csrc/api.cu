// Library-level entry points of the C ABI.
#include <mutex>
#include <vector>

#include "pvs_common.cuh"

namespace pvs {
thread_local int g_last_cuda_error = 0;
std::atomic<int64_t> g_launches{0};
thread_local bool g_pdl_chain = false;

int num_sms() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    return cached > 0 ? cached : 148;
}

int ensure_dynamic_smem(const void *func, size_t bytes) {
    struct Entry { const void *f; int dev; size_t bytes; };
    static std::mutex mu;
    static std::vector<Entry> done;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    for (const Entry &e : done)
        if (e.f == func && e.dev == dev && e.bytes >= bytes) return PVS_OK;
    int rc = cuda_call(cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                            (int)bytes));
    if (rc) return rc;
    done.push_back({func, dev, bytes});
    return PVS_OK;
}

int max_optin_smem() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&cached, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        cached_dev = dev;
    }
    return cached > 0 ? cached : 232448;
}
}  // namespace pvs

extern "C" {

int pvs_version(void) { return PVS_VERSION; }

uint32_t pvs_capabilities(void) {
    return PVS_CAP_FWD_FP32 | PVS_CAP_FWD_TCGEN05 | PVS_CAP_BWD_FP32 | PVS_CAP_FWD_FP16X2 |
           PVS_CAP_CROP | PVS_CAP_FWD_WIDE_K | PVS_CAP_POCKET;
}

const char *pvs_status_string(int status) {
    switch (status) {
        case PVS_OK: return "ok";
        case PVS_ERR_INVALID_ARG: return "invalid argument";
        case PVS_ERR_UNSUPPORTED_K:
            return "unsupported hidden width (1..64; 65..128 forward only, in a tensor-core "
                   "math mode)";
        case PVS_ERR_TOO_LARGE:
            return "complex, receptor or ligand too large for the graph kernels";
        case PVS_ERR_CUDA: return "CUDA error (see pvs_last_cuda_error)";
        case PVS_ERR_WORKSPACE: return "workspace too small";
        case PVS_ERR_UNSUPPORTED: return "configuration not supported by the kernels yet";
        default: return "unknown status";
    }
}

int pvs_last_cuda_error(void) { return pvs::g_last_cuda_error; }

int64_t pvs_launch_count(void) { return pvs::g_launches.load(std::memory_order_relaxed); }

}  // extern "C"
