// mmm_dist.cu — one large system on several B200s of one box, exact (NoCutoff) semantics.
//
// What shards: the O(N^2) pair work.  The Newton-3 kernel's work items (i-block x run of j-stages)
// are dealt to the ranks round-robin (item k of rank r is item r + k * world), every rank
// accumulates its share into its own fixed-point force planes and its own slots of the per-item
// energy array, then ONE exchange step per evaluation follows:
//     ncclAllReduce(force planes + per-item energy slots as bit patterns, uint64 sum)
// over NVLink, enqueued on the handle's stream between the pair kernel and the O(N) pass.  Integer
// sums are exact and every energy slot is written by exactly one rank (x + 0 + ... + 0), so all
// ranks hold bit-identical forces and energies — the same bits a single GPU produces — and the
// replicated O(N) state (positions, L-BFGS vectors, bonded/external pass) stays in lockstep
// without any further communication: no host round trip per iteration here either.
// What does not shard: the O(N) pass and the L-BFGS vector work (a few ms at N = 2e6 against
// seconds of pair work); they are replicated.
//
// NCCL is opened with dlopen so that the library has no load-time dependency on it (single-GPU
// users, the CPU build box).  mmm_dist_emulate runs the ranks' shares one after another on ONE
// GPU into the same accumulators: the sharding logic is testable without a second GPU.
#include <dlfcn.h>
#include <nccl.h>
#include <stdlib.h>
#include <string.h>

#include "mmm_internal.cuh"

namespace {

struct NcclApi {
  void* lib = nullptr;
  ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
  ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
  const char* (*GetErrorString)(ncclResult_t) = nullptr;
  bool ok = false;
};

NcclApi* nccl() {
  static NcclApi api;
  if (api.lib) return &api;
  // a process that already imported torch has NCCL loaded under this soname; reuse it
  api.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!api.lib) api.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!api.lib) return &api;
  api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.lib, "ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.lib, "ncclCommInitRank");
  api.AllReduce = (decltype(api.AllReduce))dlsym(api.lib, "ncclAllReduce");
  api.Broadcast = (decltype(api.Broadcast))dlsym(api.lib, "ncclBroadcast");
  api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.lib, "ncclCommDestroy");
  api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.lib, "ncclGetErrorString");
  api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.CommDestroy && api.GetErrorString;
  return &api;
}

int nccl_fail(mmm_system* h, NcclApi* a, ncclResult_t r, const char* what) {
  return mmm_fail(h, MMM_ERR_CUDA, std::string("CUDA error: NCCL ") + what + ": " + (a->GetErrorString ? a->GetErrorString(r) : "?"));
}

}  // namespace

// The exchange step: called by mmm_evaluate after the pair kernel when a communicator exists.
// ONE all-reduce: the per-item energy slots sit behind the force planes in the same allocation and
// travel as uint64 bit patterns — every slot has exactly one writer and is zero bits on the other
// ranks, and x + 0 + ... + 0 of the bit patterns is x exactly.
int mmm_dist_allreduce(mmm_system* h) {
  NcclApi* a = nccl();
  ncclComm_t comm = (ncclComm_t)h->nccl_comm;
  const size_t count = 3 * (size_t)h->npad + 4 * (size_t)h->n_items;
  MMM_CUDA(h, cudaEventRecord(h->ev_c0, h->stream));
  ncclResult_t r = a->AllReduce(h->d_facc, h->d_facc, count, ncclUint64, ncclSum, comm, h->stream);
  if (r != ncclSuccess) return nccl_fail(h, a, r, "all-reduce of the force planes and energy slots");
  MMM_CUDA(h, cudaEventRecord(h->ev_c1, h->stream));
  return MMM_OK;
}

// One work queue for all GPUs: two ticket counters in rank 0's memory, opened by every other rank
// through CUDA IPC and advanced with system-scope atomics over NVLink.  The Newton-3 kernel of every
// rank draws its items from the same counter, so a GPU that runs slower (clock, power cap) simply takes
// fewer items — no rank waits in the all-reduce for a straggler.  Which rank runs which item does not
// matter to the result (integer force accumulation, one writer per energy slot).
static int setup_global_queue(mmm_system* h, NcclApi* a) {
  h->d_gqueue = nullptr;
  h->gqueue_owner = false;
  const char* off = getenv("MMM_DIST_STATIC");
  if (off && off[0] == '1') return MMM_OK;  // static round-robin dealing (A/B timing)
  if (!a->Broadcast) return MMM_OK;
  ncclComm_t comm = (ncclComm_t)h->nccl_comm;
  cudaIpcMemHandle_t handle;
  memset(&handle, 0, sizeof(handle));
  DevBuf<int> mine;  // rank 0: the counters, handed to h->d_gqueue when every rank can reach them
  int ok = 1;
  if (h->dist_rank == 0) {
    if (mmm_reserve(h, mine, 2, "work-queue counters") != MMM_OK || cudaMemset(mine, 0, 2 * sizeof(int)) != cudaSuccess ||
        cudaIpcGetMemHandle(&handle, mine) != cudaSuccess) {
      cudaGetLastError();
      ok = 0;
    }
  }
  // ship {ok, handle} from rank 0 to everybody
  struct Msg { int ok; cudaIpcMemHandle_t handle; } msg;
  msg.ok = ok;
  msg.handle = handle;
  DevBuf<Msg> d_msg;
  int rc;
  if ((rc = mmm_reserve(h, d_msg, 1, "work-queue handle"))) return rc;
  MMM_CUDA(h, cudaMemcpyAsync(d_msg, &msg, sizeof(Msg), cudaMemcpyHostToDevice, h->stream));
  ncclResult_t r = a->Broadcast(d_msg, d_msg, sizeof(Msg), ncclChar, 0, comm, h->stream);
  if (r != ncclSuccess) return nccl_fail(h, a, r, "broadcast of the work-queue handle");
  MMM_CUDA(h, cudaMemcpyAsync(&msg, d_msg, sizeof(Msg), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  // every rank reports whether it can reach the counters; the queue is used only if all can
  int can = msg.ok;
  int* ptr = mine;
  if (can && h->dist_rank != 0) {
    void* p = nullptr;
    if (cudaIpcOpenMemHandle(&p, msg.handle, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
      cudaGetLastError();
      can = 0;
    }
    ptr = (int*)p;
  }
  DevBuf<unsigned long long> d_votes;
  if ((rc = mmm_reserve(h, d_votes, 1, "work-queue votes"))) return rc;
  const unsigned long long vote = can ? 1ull : 0ull;
  MMM_CUDA(h, cudaMemcpyAsync(d_votes, &vote, sizeof(vote), cudaMemcpyHostToDevice, h->stream));
  r = a->AllReduce(d_votes, d_votes, 1, ncclUint64, ncclSum, comm, h->stream);
  if (r != ncclSuccess) return nccl_fail(h, a, r, "all-reduce of the work-queue votes");
  unsigned long long votes = 0;
  MMM_CUDA(h, cudaMemcpyAsync(&votes, d_votes, sizeof(votes), cudaMemcpyDeviceToHost, h->stream));
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (votes == (unsigned long long)h->dist_world) {
    h->d_gqueue = h->dist_rank == 0 ? mine.release() : ptr;
    h->gqueue_owner = h->dist_rank == 0;
    h->gqueue_eval = 0;
  } else if (h->dist_rank != 0 && can && ptr) {  // somebody cannot: everybody falls back to static dealing
    cudaIpcCloseMemHandle(ptr);
  }
  return MMM_OK;
}

void mmm_dist_destroy(mmm_system* h) {
  if (h->d_gqueue) {
    if (h->gqueue_owner) cudaFree(h->d_gqueue);
    else cudaIpcCloseMemHandle(h->d_gqueue);
    h->d_gqueue = nullptr;
  }
  if (h->nccl_comm) {
    NcclApi* a = nccl();
    if (a->ok) a->CommDestroy((ncclComm_t)h->nccl_comm);
    h->nccl_comm = nullptr;
  }
}

extern "C" {

int mmm_dist_unique_id(void* out, int nbytes) {
  if (!out || nbytes < (int)sizeof(ncclUniqueId)) return MMM_ERR_ARG;
  NcclApi* a = nccl();
  if (!a->ok) return mmm_fail(nullptr, MMM_ERR_CUDA, "CUDA error: NCCL (libnccl.so.2) could not be loaded");
  ncclUniqueId id;
  ncclResult_t r = a->GetUniqueId(&id);
  if (r != ncclSuccess) return mmm_fail(nullptr, MMM_ERR_CUDA, std::string("CUDA error: NCCL ncclGetUniqueId: ") + a->GetErrorString(r));
  memcpy(out, &id, sizeof(id));
  return MMM_OK;
}

int mmm_dist_init(mmm_handle h, int rank, int world, const void* unique_id, int nbytes) {
  if (!h) return MMM_ERR_ARG;
  if (world < 1 || rank < 0 || rank >= world) return mmm_fail(h, MMM_ERR_ARG, "mmm_dist_init: need 0 <= rank < world");
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  mmm_dist_destroy(h);
  h->dist_emulate = false;
  h->dist_rank = rank;
  h->dist_world = world;
  if (world > 1) {
    if (!unique_id || nbytes < (int)sizeof(ncclUniqueId)) return mmm_fail(h, MMM_ERR_ARG, "mmm_dist_init: unique id missing");
    NcclApi* a = nccl();
    if (!a->ok) return mmm_fail(h, MMM_ERR_CUDA, "CUDA error: NCCL (libnccl.so.2) could not be loaded");
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof(id));
    ncclComm_t comm;
    ncclResult_t r = a->CommInitRank(&comm, world, id, rank);
    if (r != ncclSuccess) return nccl_fail(h, a, r, "ncclCommInitRank");
    h->nccl_comm = comm;
    if (!h->ev_c0) { cudaEventCreate(&h->ev_c0); cudaEventCreate(&h->ev_c1); }
    int rc = setup_global_queue(h, a);
    if (rc) return rc;
  }
  h->scratch_sig = -2;  // re-size the scratch (local energy slots)
  return MMM_OK;
}

int mmm_dist_queue_mode(mmm_handle h) { return (h && h->d_gqueue) ? 1 : 0; }

int mmm_dist_last_exchange_ms(mmm_handle h, float* ms_out) {
  if (!h || !ms_out) return MMM_ERR_ARG;
  *ms_out = 0.f;
  if (!h->nccl_comm || !h->ev_c0) return MMM_OK;
  cudaSetDevice(h->device);
  MMM_CUDA(h, cudaStreamSynchronize(h->stream));
  if (cudaEventElapsedTime(ms_out, h->ev_c0, h->ev_c1) != cudaSuccess) { cudaGetLastError(); *ms_out = 0.f; }
  return MMM_OK;
}

int mmm_dist_emulate(mmm_handle h, int world) {
  if (!h) return MMM_ERR_ARG;
  if (world < 1) return mmm_fail(h, MMM_ERR_ARG, "mmm_dist_emulate: world must be >= 1");
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  mmm_dist_destroy(h);
  h->dist_rank = 0;
  h->dist_world = world;
  h->dist_emulate = world > 1;
  h->scratch_sig = -2;
  return MMM_OK;
}

}  // extern "C"
