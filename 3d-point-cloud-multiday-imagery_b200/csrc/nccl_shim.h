// Minimal run-time binding to NCCL (dlopen) so that libmdkm.so has no link-time dependency:
// the library loads on a CPU-only box (symbol-export tests) and, in a process that already
// imported torch, reuses the libnccl.so.2 torch loaded.  Only the handful of calls the
// K x 4 partial-sum exchange needs.
#pragma once
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stddef.h>

namespace mdkm {

typedef struct ncclComm* ncclComm_t;
typedef struct { char internal[128]; } ncclUniqueId;
typedef int ncclResult_t;
// values from nccl.h (stable across 2.x)
enum { kNcclUint8 = 1, kNcclUint32 = 3, kNcclInt64 = 4, kNcclUint64 = 5, kNcclFloat32 = 7, kNcclFloat64 = 8 };
enum { kNcclSum = 0, kNcclMax = 2, kNcclMin = 3 };

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  ncclResult_t (*GetVersion)(int*) = nullptr;
  bool ok = false;
};

inline NcclApi& nccl_api() {
  static NcclApi api;
  if (api.ok || api.lib) return api;
  const char* env = getenv("MDKM_NCCL_LIB");
  const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
  for (const char* nm : names) {
    if (!nm || !*nm) continue;
    void* l = dlopen(nm, RTLD_NOW | RTLD_NOLOAD);  // already in the process (torch)?
    if (!l) l = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
    if (l) { api.lib = l; break; }
  }
  if (!api.lib) return api;
  api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
  api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
  api.AllReduce = (decltype(api.AllReduce))dlsym(api.lib, "ncclAllReduce");
  api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
  api.GetVersion = (decltype(api.GetVersion))dlsym(api.lib, "ncclGetVersion");
  api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce;
  return api;
}

}  // namespace mdkm
