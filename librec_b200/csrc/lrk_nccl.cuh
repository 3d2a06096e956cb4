// NCCL, dlopen'ed lazily so that the single-GPU path has no NCCL dependency (DSGD ranks: staging.cuh, dsgd.cuh).
#pragma once
#include "lrk_common.cuh"
#include <nccl.h>
#include <dlfcn.h>

struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
};

static NcclApi* nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return api.lib ? &api : nullptr;
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) { api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (api.lib) break; }
    if (!api.lib) return nullptr;
#define LRK_SYM(field, sym) *(void**)(&api.field) = dlsym(api.lib, sym); if (!api.field) { api.lib = nullptr; return nullptr; }
    LRK_SYM(GetUniqueId, "ncclGetUniqueId") LRK_SYM(CommInitRank, "ncclCommInitRank") LRK_SYM(CommDestroy, "ncclCommDestroy")
    LRK_SYM(Send, "ncclSend") LRK_SYM(Recv, "ncclRecv") LRK_SYM(AllReduce, "ncclAllReduce") LRK_SYM(AllGather, "ncclAllGather")
    LRK_SYM(GroupStart, "ncclGroupStart") LRK_SYM(GroupEnd, "ncclGroupEnd") LRK_SYM(GetErrorString, "ncclGetErrorString")
#undef LRK_SYM
    return &api;
}

#define LRK_NCCL(h, call)                                                                                         \
    do {                                                                                                          \
        ncclResult_t r__ = (call);                                                                                \
        if (r__ != ncclSuccess) return lrk_fail((h), LRK_ERR_NCCL, #call, nccl_api()->GetErrorString(r__), __FILE__, __LINE__); \
    } while (0)
