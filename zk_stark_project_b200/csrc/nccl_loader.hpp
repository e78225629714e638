// Lazy NCCL binding for the column-sharded multi-GPU proof (zkb_mg_*).  Included by zkb200.cu after CudaError is defined.
#pragma once
#include <dlfcn.h>
#include <nccl.h>
#include <string>

namespace zkb {

// NCCL is resolved lazily (dlopen) so the single-GPU path never depends on it; if the process already loaded an NCCL
// with the same SONAME (e.g. torch's), that copy is reused.
struct NcclApi {
    void* h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    void load() {
        if (h) return;
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) { h = dlopen(name, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
        if (!h) throw CudaError(std::string("cannot load NCCL: ") + dlerror());
        auto sym = [&](const char* n) { void* f = dlsym(h, n); if (!f) throw CudaError(std::string("NCCL symbol missing: ") + n); return f; };
        GetUniqueId = (decltype(GetUniqueId))sym("ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))sym("ncclCommInitRank");
        CommDestroy = (decltype(CommDestroy))sym("ncclCommDestroy");
        GroupStart = (decltype(GroupStart))sym("ncclGroupStart");
        GroupEnd = (decltype(GroupEnd))sym("ncclGroupEnd");
        Send = (decltype(Send))sym("ncclSend");
        Recv = (decltype(Recv))sym("ncclRecv");
        AllGather = (decltype(AllGather))sym("ncclAllGather");
        AllReduce = (decltype(AllReduce))sym("ncclAllReduce");
        GetErrorString = (decltype(GetErrorString))sym("ncclGetErrorString");
    }
};
static NcclApi g_nccl;
#define NK(call)                                                                                                        \
    do {                                                                                                                \
        ncclResult_t r_ = (call);                                                                                       \
        if (r_ != ncclSuccess) throw CudaError(std::string(#call) + " failed: " + g_nccl.GetErrorString(r_));           \
    } while (0)

}  // namespace zkb
