// Data-parallel helpers of the train step (SURVEY.md 8e): the collectives between the train-step phases,
// issued with NCCL on the caller's stream.  The reference has no distributed code at all (train.py is
// single-device); these are the exchanges that make the row-sharded step equal to the single-device step:
//   ShiftBounds batch min/max (bijectors.py:250-252)  -> one all-reduce(min) over [min | -max]
//   BatchNorm batch moments, forward and backward     -> all-reduce(sum) of 2F doubles
//   parameter gradients (train.py:82)                 -> all-reduce(sum) of the flat gradient, bucketed per coupling
// libnccl is resolved at run time (dlopen; the copy the host process already loaded wins), so the library
// itself keeps linking against the CUDA runtime only.
#include "zf_common.cuh"

#include <dlfcn.h>
#include <mutex>
#include <string.h>

#if __has_include(<nccl.h>)
#include <nccl.h>
#else
extern "C" {
typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef enum { ncclSuccess = 0 } ncclResult_t;
typedef enum { ncclInt8 = 0, ncclUint8 = 1, ncclInt32 = 2, ncclUint32 = 3, ncclInt64 = 4, ncclUint64 = 5,
               ncclFloat16 = 6, ncclFloat32 = 7, ncclFloat64 = 8 } ncclDataType_t;
typedef enum { ncclSum = 0, ncclProd = 1, ncclMax = 2, ncclMin = 3 } ncclRedOp_t;
}
#endif

namespace zf {

struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*CommCount)(const ncclComm_t, int*) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

static int nccl_api(const NcclApi** out) {
    static std::mutex mu;
    static NcclApi api;
    static bool tried = false, ok = false;
    std::lock_guard<std::mutex> lock(mu);
    if (!tried) {
        tried = true;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {   // the copy already mapped into the process (e.g. the host framework's) first
            api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) {
            const char* env = getenv("ZF_NCCL_LIBRARY");
            if (env && env[0]) api.handle = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
        }
        for (const char* n : names) {
            if (api.handle) break;
            api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        }
        if (api.handle) {
            auto sym = [&](const char* s) { return dlsym(api.handle, s); };
            api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
            api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
            api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
            api.CommCount = reinterpret_cast<decltype(api.CommCount)>(sym("ncclCommCount"));
            api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
            api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
            api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
            api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
            ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.CommCount && api.AllReduce &&
                 api.GetErrorString;
        }
    }
    if (!ok) return fail(ZF_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded (set ZF_NCCL_LIBRARY): %s",
                         api.handle ? "missing symbols" : dlerror());
    *out = &api;
    return ZF_OK;
}

#define ZF_NCCL_CHECK(api, expr)                                                                   \
    do {                                                                                           \
        ncclResult_t _r = (expr);                                                                  \
        if (_r != ncclSuccess)                                                                     \
            return zf::fail(ZF_ERR_CUDA, "%s failed: %s", #expr, (api)->GetErrorString(_r));      \
    } while (0)

// max half of [min | max] <-> its negation, so that one all-reduce(min) serves both halves
__global__ void negate_tail_kernel(float* v, int D) {
    const int i = threadIdx.x;
    if (i < D) v[D + i] = -v[D + i];
}

int dp_allreduce(cudaStream_t st, void* comm, void* buf, long long n, int is_f64, int op /*0 sum, 1 min*/) {
    if (!comm || n <= 0) return ZF_OK;
    const NcclApi* api;
    if (int rc = nccl_api(&api)) return rc;
    ZF_NCCL_CHECK(api, api->AllReduce(buf, buf, (size_t)n, is_f64 ? ncclFloat64 : ncclFloat32, op ? ncclMin : ncclSum,
                                      (ncclComm_t)comm, st));
    count_launch();
    return ZF_OK;
}

}  // namespace zf

using namespace zf;

extern "C" int zf_dp_unique_id(void* id_out) {
    ZF_REQUIRE(id_out != nullptr, "dp_unique_id: null argument");
    const NcclApi* api;
    if (int rc = nccl_api(&api)) return rc;
    ncclUniqueId id;
    ZF_NCCL_CHECK(api, api->GetUniqueId(&id));
    static_assert(sizeof(ncclUniqueId) == ZF_DP_UNIQUE_ID_BYTES, "ncclUniqueId size");
    memcpy(id_out, &id, sizeof(id));
    return ZF_OK;
}

extern "C" int zf_dp_comm_create(const void* id, int32_t rank, int32_t world, void** comm_out) {
    ZF_REQUIRE(id && comm_out && world >= 1 && rank >= 0 && rank < world, "dp_comm_create: bad argument");
    const NcclApi* api;
    if (int rc = nccl_api(&api)) return rc;
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof(uid));
    ncclComm_t comm = nullptr;
    ZF_NCCL_CHECK(api, api->CommInitRank(&comm, world, uid, rank));
    *comm_out = comm;
    return ZF_OK;
}

extern "C" int zf_dp_comm_destroy(void* comm) {
    if (!comm) return ZF_OK;
    const NcclApi* api;
    if (int rc = nccl_api(&api)) return rc;
    ZF_NCCL_CHECK(api, api->CommDestroy((ncclComm_t)comm));
    return ZF_OK;
}

extern "C" int zf_dp_comm_size(void* comm, int32_t* world_out) {
    ZF_REQUIRE(world_out != nullptr, "dp_comm_size: null argument");
    if (!comm) { *world_out = 1; return ZF_OK; }
    const NcclApi* api;
    if (int rc = nccl_api(&api)) return rc;
    int n = 0;
    ZF_NCCL_CHECK(api, api->CommCount((ncclComm_t)comm, &n));
    *world_out = n;
    return ZF_OK;
}

extern "C" int zf_dp_allreduce_sum_f32(void* stream, void* comm, float* buf, int64_t n) {
    ZF_REQUIRE(buf || n == 0, "dp_allreduce_sum_f32: null buffer");
    return dp_allreduce((cudaStream_t)stream, comm, buf, n, 0, 0);
}

extern "C" int zf_dp_allreduce_sum_f64(void* stream, void* comm, double* buf, int64_t n) {
    ZF_REQUIRE(buf || n == 0, "dp_allreduce_sum_f64: null buffer");
    return dp_allreduce((cudaStream_t)stream, comm, buf, n, 1, 0);
}

extern "C" int zf_dp_allreduce_minmax_f32(void* stream, void* comm, float* minmax, int32_t D) {
    ZF_REQUIRE(minmax && D >= 1 && D <= ZF_MAX_DIM, "dp_allreduce_minmax_f32: bad argument");
    if (!comm) return ZF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    negate_tail_kernel<<<1, ZF_MAX_DIM, 0, st>>>(minmax, D);
    count_launch();
    if (int rc = dp_allreduce(st, comm, minmax, 2 * D, 0, 1)) return rc;
    negate_tail_kernel<<<1, ZF_MAX_DIM, 0, st>>>(minmax, D);
    count_launch();
    ZF_CUDA_CHECK(cudaGetLastError());
    return ZF_OK;
}
