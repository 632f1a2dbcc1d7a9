// nccl_api.h — the NCCL entry points the library uses, resolved once by nccl_load() (xalm_cuda.cu) from the libnccl that
// dlopen finds: single-GPU users need no libnccl at all, and inside a torch process the already-loaded libnccl.so.2 is the
// one dlopen returns.  Shared by the decode exchange (xalm_cuda.cu) and the batched prefill (prefill.cu).
#pragma once
#include <cuda_runtime.h>
#include <nccl.h>

namespace xalm {

struct NcclApi {
	void* h = nullptr;
	ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
	ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
	ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*ReduceScatter)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
	ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
	const char* (*GetErrorString)(ncclResult_t) = nullptr;
};
extern NcclApi g_nccl;
int nccl_load();

#define XALM_NCCL_CHECK(expr)                                                                                     \
	do {                                                                                                          \
		ncclResult_t _r = (expr);                                                                                 \
		if (_r != ncclSuccess) return set_error(XALM_ERR_COMM, "%s failed: %s", #expr, g_nccl.GetErrorString(_r)); \
	} while (0)

} // namespace xalm
