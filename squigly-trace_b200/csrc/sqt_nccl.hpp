// sqt_nccl.hpp -- NCCL reached through dlopen, so that the single-GPU path has no NCCL dependency at all.
// Only the handful of entry points the render path uses (ncclReduce of the accumulation buffers -- and moments and
// sample counts --, a few-word ncclAllReduce with which the ranks agree that all of them can enter it or sum their
// active pixels, ncclCommAbort for the case they cannot).
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <string>

typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*CommAbort)(ncclComm_t) = nullptr;
    ncclResult_t (*Reduce)(const void *, void *, size_t, int, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    std::string err;
};
inline NcclApi *nccl_api() {
    static NcclApi api;
    static bool tried = false;
    if (tried) return &api;
    tried = true;
    const char *names[] = {"libnccl.so.2", "libnccl.so", "/usr/lib/x86_64-linux-gnu/libnccl.so.2"};
    for (const char *n : names) { api.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (api.lib) break; }
    if (!api.lib) { api.err = std::string("cannot dlopen libnccl.so.2: ") + dlerror(); return &api; }
#define SQT_SYM(field, name) *(void **)(&api.field) = dlsym(api.lib, name); if (!api.field) { api.err = "NCCL symbol missing: " name; api.lib = nullptr; return &api; }
    SQT_SYM(GetUniqueId, "ncclGetUniqueId") SQT_SYM(CommInitRank, "ncclCommInitRank") SQT_SYM(CommInitAll, "ncclCommInitAll")
    SQT_SYM(CommDestroy, "ncclCommDestroy") SQT_SYM(CommAbort, "ncclCommAbort") SQT_SYM(Reduce, "ncclReduce") SQT_SYM(AllReduce, "ncclAllReduce")
    SQT_SYM(GroupStart, "ncclGroupStart") SQT_SYM(GroupEnd, "ncclGroupEnd") SQT_SYM(GetErrorString, "ncclGetErrorString")
#undef SQT_SYM
    return &api;
}
static const int kNcclInt32 = 2, kNcclInt64 = 4, kNcclFloat32 = 7, kNcclSum = 0, kNcclMax = 2;
