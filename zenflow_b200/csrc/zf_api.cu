// C-ABI plumbing: thread-local error message, launch counter, per-device attribute cache, shared-memory opt-in.
#include "zf_common.cuh"

#include <map>
#include <mutex>
#include <string.h>

namespace zf {

static thread_local char g_err[512] = "";
static thread_local long long g_launches = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

void count_launch() { ++g_launches; }

int get_device_info(DeviceInfo* out) {
    static std::mutex mu;
    static DeviceInfo cache[64];
    static bool have[64] = {false};
    int dev = 0;
    ZF_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(ZF_ERR_UNSUPPORTED, "device ordinal %d out of range", dev);
    std::lock_guard<std::mutex> lock(mu);
    if (!have[dev]) {
        DeviceInfo di{};
        di.device = dev;
        ZF_CUDA_CHECK(cudaDeviceGetAttribute(&di.sm_count, cudaDevAttrMultiProcessorCount, dev));
        ZF_CUDA_CHECK(cudaDeviceGetAttribute(&di.max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        ZF_CUDA_CHECK(cudaDeviceGetAttribute(&di.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
        ZF_CUDA_CHECK(cudaDeviceGetAttribute(&di.cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
        if (di.cc_major != 10)
            return fail(ZF_ERR_UNSUPPORTED, "zenflow_b200 is built for sm_100a only (device is sm_%d%d)",
                        di.cc_major, di.cc_minor);
        cache[dev] = di;
        have[dev] = true;
    }
    *out = cache[dev];
    return ZF_OK;
}

int smem_optin(const void* fn, size_t bytes) {
    static std::mutex mu;
    static std::map<std::pair<const void*, int>, size_t> done;
    int dev = 0;
    ZF_CUDA_CHECK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    size_t& have = done[{fn, dev}];
    if (have < bytes) {
        ZF_CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        have = bytes;
    }
    return ZF_OK;
}

}  // namespace zf

extern "C" int32_t zf_abi_version(void) { return ZF_ABI_VERSION; }
extern "C" const char* zf_last_error(void) { return zf::g_err; }
extern "C" int64_t zf_launch_count(void) { return zf::g_launches; }
extern "C" void zf_launch_count_add(int64_t n) { zf::g_launches += n; }
