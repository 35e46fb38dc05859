// Run-time binding of NCCL for the multi-GPU entry points of the C ABI (locreg_comm_*, locreg_relocalise_sharded,
// locreg_relocalise_loam_sharded, locreg_relocalise_staged_sharded, locreg_align_batch_sharded).  liblocreg.so carries
// no DT_NEEDED on libnccl: a single-GPU user (slam_demo's tracking loop) needs no NCCL, and a process that already holds
// a copy (torch ships its own libnccl.so.2) must not get a second one.  The first use looks for a loaded libnccl.so.2
// (RTLD_NOLOAD), then for the system's.
#pragma once
#include <dlfcn.h>
#include <nccl.h>

#include <mutex>
#include <string>

namespace locreg {

struct NcclApi {
    ncclResult_t (*GetVersion)(int*) = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    std::string why;  // empty when bound
    bool ok() const { return why.empty(); }
};

inline const NcclApi& nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!lib) { api.why = std::string("libnccl.so.2 not found: ") + dlerror(); return; }
        auto sym = [&](const char* name) -> void* {
            void* p = dlsym(lib, name);
            if (!p && api.why.empty()) api.why = std::string("libnccl.so.2 lacks ") + name;
            return p;
        };
        api.GetVersion = reinterpret_cast<decltype(api.GetVersion)>(sym("ncclGetVersion"));
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(sym("ncclAllReduce"));
        api.Broadcast = reinterpret_cast<decltype(api.Broadcast)>(sym("ncclBroadcast"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(sym("ncclGroupStart"));
        api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(sym("ncclGroupEnd"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
    });
    return api;
}

struct NcclError : std::runtime_error {
    using std::runtime_error::runtime_error;
};
#define LR_NCCL(expr)                                                                                     \
    do {                                                                                                  \
        ncclResult_t r_ = (expr);                                                                         \
        if (r_ != ncclSuccess)                                                                            \
            throw ::locreg::NcclError(std::string(#expr) + ": " + ::locreg::nccl_api().GetErrorString(r_)); \
    } while (0)

}  // namespace locreg
