// replicate.hpp -- the one collective of the path (SURVEY 8e): after the table is built on one GPU its raw slot array
// is broadcast ONCE over NVLink / NVSwitch with ncclBroadcast, issued by the library itself; every receiver then
// derives its successor tables locally.  No per-read or per-batch communication exists anywhere.
//
// NCCL is bound at run time (dlopen "libnccl.so.2"): inside a torchrun process that is the copy torch has already
// loaded, in the stand-alone `talc` command line the system one.  The library has no link-time dependency on it;
// when it is absent talc_table_replicate falls back to peer copies and says so.
// Included at the end of talc_b200.cu (same translation unit as the context).
#pragma once
#include <dlfcn.h>

namespace nccl_dyn {
typedef struct ncclComm* ncclComm_t;
struct ncclUniqueId { char internal[128]; };
typedef int ncclResult_t;
enum { ncclUint8 = 1 };
struct Api {
  void* h = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*GroupStart)() = nullptr;
  ncclResult_t (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok() const { return h && GetUniqueId && CommInitRank && CommInitAll && CommDestroy && Broadcast && GroupStart && GroupEnd; }
};
static Api& api() {
  static Api a;
  static bool tried = false;
  if (!tried) {
    tried = true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
      a.h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
      if (a.h) break;
    }
    if (a.h) {
      a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(a.h, "ncclGetUniqueId");
      a.CommInitRank = (decltype(a.CommInitRank))dlsym(a.h, "ncclCommInitRank");
      a.CommInitAll = (decltype(a.CommInitAll))dlsym(a.h, "ncclCommInitAll");
      a.CommDestroy = (decltype(a.CommDestroy))dlsym(a.h, "ncclCommDestroy");
      a.Broadcast = (decltype(a.Broadcast))dlsym(a.h, "ncclBroadcast");
      a.GroupStart = (decltype(a.GroupStart))dlsym(a.h, "ncclGroupStart");
      a.GroupEnd = (decltype(a.GroupEnd))dlsym(a.h, "ncclGroupEnd");
      a.GetErrorString = (decltype(a.GetErrorString))dlsym(a.h, "ncclGetErrorString");
    }
  }
  return a;
}
}  // namespace nccl_dyn

extern "C" {

int talc_nccl_available(void) { return nccl_dyn::api().ok() ? 1 : 0; }

// 128 bytes that rank 0 hands to the other ranks by any means (bench.py: torch.distributed broadcast)
int talc_nccl_unique_id(uint8_t id[128]) {
  if (!id) return TALC_ERR_ARG;
  auto& N = nccl_dyn::api();
  if (!N.ok()) return TALC_ERR_NCCL;
  nccl_dyn::ncclUniqueId u;
  if (N.GetUniqueId(&u) != 0) return TALC_ERR_NCCL;
  memcpy(id, u.internal, 128);
  return TALC_OK;
}

// Multi-process replication (one process per GPU): every rank calls this with the same id.  The root's sealed table
// is broadcast -- first its geometry (capacity, entries, provenance), then the slot array with ONE ncclBroadcast -- and
// every other rank allocates, receives and seals.  broadcast_ms = device time of the slot-array broadcast.
int talc_table_broadcast(talc_ctx* c, const uint8_t id[128], int rank, int world, int root, double* broadcast_ms) {
  if (!c || !id || world < 1 || rank < 0 || rank >= world || root < 0 || root >= world) return TALC_ERR_ARG;
  auto& N = nccl_dyn::api();
  if (!N.ok()) { c->err = "NCCL (libnccl.so.2) could not be loaded"; return TALC_ERR_NCCL; }
  if (rank == root && !c->tableReady) { c->err = "the root has no table to broadcast"; return TALC_ERR_NO_TABLE; }
  CUDA_TRY(c, cudaSetDevice(c->device));
  nccl_dyn::ncclUniqueId u;
  memcpy(u.internal, id, 128);
  nccl_dyn::ncclComm_t comm = nullptr;
  int r = N.CommInitRank(&comm, world, u, rank);
  if (r != 0) { c->err = std::string("ncclCommInitRank: ") + (N.GetErrorString ? N.GetErrorString(r) : "error"); return TALC_ERR_NCCL; }
  u64* dMeta = nullptr;
  u64 hMeta[8] = {c->capacity, c->nEntries, c->provJunctions, c->provDumpSize, c->provDumpMtime, c->provJuncSize, c->provJuncMtime, c->provFlags};
  int rc = TALC_OK;
  do {
    if (cudaMalloc((void**)&dMeta, sizeof(hMeta)) != cudaSuccess) { rc = TALC_ERR_CUDA; break; }
    if (rank == root) cudaMemcpyAsync(dMeta, hMeta, sizeof(hMeta), cudaMemcpyHostToDevice, c->stream);
    if (N.Broadcast(dMeta, dMeta, sizeof(hMeta), nccl_dyn::ncclUint8, root, comm, c->stream) != 0) { rc = TALC_ERR_NCCL; break; }
    if (cudaMemcpyAsync(hMeta, dMeta, sizeof(hMeta), cudaMemcpyDeviceToHost, c->stream) != cudaSuccess ||
        cudaStreamSynchronize(c->stream) != cudaSuccess) { rc = TALC_ERR_CUDA; break; }
    if (rank != root) {
      rc = talc_table_alloc(c, hMeta[0]);
      if (rc) break;
      c->provJunctions = (u32)hMeta[2];
      c->provFlags = (u32)hMeta[7];
      c->provDumpSize = hMeta[3]; c->provDumpMtime = hMeta[4]; c->provJuncSize = hMeta[5]; c->provJuncMtime = hMeta[6];
    }
    cudaEventRecord(c->ev[6], c->stream);
    if (N.Broadcast(c->slots, c->slots, (size_t)hMeta[0] * sizeof(Slot), nccl_dyn::ncclUint8, root, comm, c->stream) != 0) { rc = TALC_ERR_NCCL; break; }
    cudaEventRecord(c->ev[7], c->stream);
    if (cudaStreamSynchronize(c->stream) != cudaSuccess) { rc = TALC_ERR_CUDA; break; }
    float ms = 0;
    cudaEventElapsedTime(&ms, c->ev[6], c->ev[7]);
    if (broadcast_ms) *broadcast_ms = ms;
    if (rank != root) rc = talc_table_seal(c, hMeta[1]);
  } while (0);
  if (dMeta) cudaFree(dMeta);
  N.CommDestroy(comm);
  if (rc == TALC_ERR_NCCL) c->err = "ncclBroadcast failed";
  if (rc == TALC_ERR_CUDA && c->err.empty()) c->err = "CUDA error during the table broadcast";
  return rc;
}

// Single-process replication (the `talc --gpus N` command line): ctxs[0] holds the sealed table, ctxs[1..n) receive it
// through ONE grouped ncclBroadcast over a communicator made with ncclCommInitAll.  used_nccl (may be NULL) tells
// whether NCCL carried it or the fallback (cudaMemcpyPeer per replica) did.
int talc_table_replicate(talc_ctx** ctxs, int n, double* broadcast_ms, int* used_nccl) {
  if (!ctxs || n < 1 || !ctxs[0] || !ctxs[0]->tableReady) return TALC_ERR_ARG;
  if (broadcast_ms) *broadcast_ms = 0;
  if (used_nccl) *used_nccl = 0;
  if (n == 1) return TALC_OK;
  talc_ctx* src = ctxs[0];
  auto& N = nccl_dyn::api();
  if (!N.ok()) {
    for (int i = 1; i < n; ++i) {
      const int rc = talc_table_copy(ctxs[i], src);
      if (rc) return rc;
    }
    return TALC_OK;
  }
  std::vector<int> devs(n);
  for (int i = 0; i < n; ++i) devs[i] = ctxs[i]->device;
  for (int i = 1; i < n; ++i) {
    const int rc = talc_table_alloc(ctxs[i], src->capacity);
    if (rc) return rc;
    ctxs[i]->provJunctions = src->provJunctions;
    ctxs[i]->provFlags = src->provFlags;
    ctxs[i]->provDumpSize = src->provDumpSize; ctxs[i]->provDumpMtime = src->provDumpMtime;
    ctxs[i]->provJuncSize = src->provJuncSize; ctxs[i]->provJuncMtime = src->provJuncMtime;
  }
  std::vector<nccl_dyn::ncclComm_t> comms(n, nullptr);
  if (N.CommInitAll(comms.data(), n, devs.data()) != 0) { src->err = "ncclCommInitAll failed"; return TALC_ERR_NCCL; }
  int rc = TALC_OK;
  cudaSetDevice(src->device);
  cudaEventRecord(src->ev[6], src->stream);
  N.GroupStart();
  for (int i = 0; i < n; ++i) {
    cudaSetDevice(ctxs[i]->device);
    if (N.Broadcast(ctxs[i]->slots, ctxs[i]->slots, (size_t)src->capacity * sizeof(Slot),
                    nccl_dyn::ncclUint8, 0, comms[i], ctxs[i]->stream) != 0)
      rc = TALC_ERR_NCCL;
  }
  if (N.GroupEnd() != 0) rc = TALC_ERR_NCCL;
  cudaSetDevice(src->device);
  cudaEventRecord(src->ev[7], src->stream);
  for (int i = 0; i < n; ++i) {
    cudaSetDevice(ctxs[i]->device);
    if (cudaStreamSynchronize(ctxs[i]->stream) != cudaSuccess) rc = TALC_ERR_CUDA;
  }
  if (rc == TALC_OK && broadcast_ms) {
    float ms = 0;
    cudaEventElapsedTime(&ms, src->ev[6], src->ev[7]);
    *broadcast_ms = ms;
  }
  for (auto cm : comms)
    if (cm) N.CommDestroy(cm);
  if (rc != TALC_OK) { src->err = "ncclBroadcast of the k-mer table failed"; return rc; }
  for (int i = 1; i < n; ++i) {
    rc = talc_table_seal(ctxs[i], src->nEntries);
    if (rc) return rc;
  }
  if (used_nccl) *used_nccl = 1;
  return TALC_OK;
}

}  // extern "C"
