// nccl_dyn.h — NCCL resolved at run time with dlopen, so that the single-GPU library has no NCCL dependency
// and a multi-rank process shares whichever libnccl.so.2 its host (e.g. torch) already loaded.
// Only the stable subset of the NCCL 2.x C ABI needed for halo send/recv and scalar all-reduce is declared.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stddef.h>

namespace wafer {

struct NcclUniqueId { char internal[128]; };
typedef struct ncclComm* NcclComm;
enum { kNcclSuccess = 0, kNcclUint64 = 5, kNcclFloat64 = 8, kNcclSum = 0 };

struct NcclApi {
    void* handle = nullptr;
    int (*GetUniqueId)(NcclUniqueId*) = nullptr;
    int (*CommInitRank)(NcclComm*, int, NcclUniqueId, int) = nullptr;
    int (*CommDestroy)(NcclComm) = nullptr;
    int (*Send)(const void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    int (*GetVersion)(int*) = nullptr;

    // returns nullptr on success, else a static description of what failed
    const char* load() {
        if (handle) return nullptr;
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (handle) break;
        }
        if (!handle) return "dlopen(libnccl.so.2) failed";
#define WAFER_NCCL_SYM(field, sym)                                   \
    field = reinterpret_cast<decltype(field)>(dlsym(handle, sym));  \
    if (!field) return "missing NCCL symbol " sym;
        WAFER_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
        WAFER_NCCL_SYM(CommInitRank, "ncclCommInitRank")
        WAFER_NCCL_SYM(CommDestroy, "ncclCommDestroy")
        WAFER_NCCL_SYM(Send, "ncclSend")
        WAFER_NCCL_SYM(Recv, "ncclRecv")
        WAFER_NCCL_SYM(AllReduce, "ncclAllReduce")
        WAFER_NCCL_SYM(GroupStart, "ncclGroupStart")
        WAFER_NCCL_SYM(GroupEnd, "ncclGroupEnd")
        WAFER_NCCL_SYM(GetErrorString, "ncclGetErrorString")
        WAFER_NCCL_SYM(GetVersion, "ncclGetVersion")
#undef WAFER_NCCL_SYM
        return nullptr;
    }
};

inline NcclApi& nccl_api() {
    static NcclApi api;
    return api;
}

}  // namespace wafer
