// engine_comm.cu — sharded pools: NCCL binding, fi_epp_comm_init, peer-memory exchange.
#include "engine.h"
#include <dlfcn.h>
#include <unistd.h>

namespace {

// ---- minimal NCCL binding through dlopen (the torch-bundled or the system libnccl.so.2) ----
typedef struct {
  char internal[128];
} ncclUniqueId;
enum { ncclSuccess = 0 };
enum { ncclInt8 = 0, ncclChar = 0, ncclUint8 = 1 };
struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(ncclUniqueId*) = nullptr;
  int (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
  int (*CommDestroy)(ncclComm_t) = nullptr;
  int (*AllGather)(const void*, void*, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool load(std::string* err) {
    if (lib) return true;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* n : names) {
      lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
      if (lib) break;
    }
    if (!lib) {
      *err = std::string("dlopen libnccl.so.2 failed: ") + dlerror();
      return false;
    }
    GetUniqueId = (decltype(GetUniqueId))dlsym(lib, "ncclGetUniqueId");
    CommInitRank = (decltype(CommInitRank))dlsym(lib, "ncclCommInitRank");
    CommDestroy = (decltype(CommDestroy))dlsym(lib, "ncclCommDestroy");
    AllGather = (decltype(AllGather))dlsym(lib, "ncclAllGather");
    GetErrorString = (decltype(GetErrorString))dlsym(lib, "ncclGetErrorString");
    if (!GetUniqueId || !CommInitRank || !CommDestroy || !AllGather) {
      *err = "libnccl is missing a required symbol";
      return false;
    }
    return true;
  }
};
NcclApi g_nccl;
std::mutex g_nccl_mu;

}  // namespace

void fi::comm_destroy(ncclComm_t c) { if (g_nccl.CommDestroy) g_nccl.CommDestroy(c); }

namespace fi {

int nccl_allgather(fi_epp* h, ncclComm_t comm, const void* send, void* recv, size_t bytes, cudaStream_t s) {
  int rc = g_nccl.AllGather(send, recv, bytes, ncclInt8, comm, s);
  if (rc != ncclSuccess)
    return fail(h, FI_ERR_COMM, std::string("ncclAllGather: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error"));
  return FI_OK;
}

// Peer-memory exchange set-up (sharded mode): allocate this rank's buffer, exchange its IPC handle over
// the NCCL communicator, map every peer's buffer.  Falls back to the NCCL all-gather path (px.enabled = 0)
// when FI_EPP_EXCHANGE=nccl, when there are more than FI_MAX_RANKS ranks, or when any rank cannot map a peer.
struct XchgBlob {
  cudaIpcMemHandle_t handle;
  uint64_t ptr;
  int64_t pid;
  int32_t device;
  int32_t ok;
  uint8_t pad[40];
};
static_assert(sizeof(XchgBlob) == 128, "XchgBlob size");

int setup_peer_exchange(fi_epp* h, Shard& sh, uint32_t rank, uint32_t world) {
  const char* mode = std::getenv("FI_EPP_EXCHANGE");
  const bool want = !(mode && std::strcmp(mode, "nccl") == 0) && world <= (uint32_t)FI_MAX_RANKS;
  const uint64_t R = h->cfg.max_batch;
  auto up = [](uint64_t v) { return (v + 255) & ~255ull; };
  PeerXchg px{};
  px.world = world;
  px.rank = rank;
  uint64_t off = 0;
  for (int par = 0; par < 2; ++par) {  // tagged 64-bit words (kernels.cuh PeerXchg)
    px.off_pick[par] = off;
    off = up(off + (uint64_t)world * R * h->P * 4 * sizeof(uint64_t));
  }
  XchgBlob mine{};
  mine.ok = 0;
  if (want && dev_alloc(sh.d_xchg, off) == cudaSuccess && cudaMemset(sh.d_xchg.get(), 0, off) == cudaSuccess &&
      host_alloc(sh.h_xerr, sizeof(uint32_t), cudaHostAllocMapped) == cudaSuccess &&
      cudaIpcGetMemHandle(&mine.handle, sh.d_xchg.get()) == cudaSuccess) {
    mine.ok = 1;
  }
  cudaGetLastError();
  mine.ptr = (uint64_t)(uintptr_t)sh.d_xchg.get();
  mine.pid = (int64_t)getpid();
  mine.device = h->cfg.device;
  // round 1: handles; round 2: "I mapped every peer" votes.  Both ride the NCCL communicator.
  DevPtr<XchgBlob> d_blobs;
  FI_CUDA(dev_alloc(d_blobs, (size_t)(world + 1) * sizeof(XchgBlob)));
  std::vector<XchgBlob> all(world);
  auto gather = [&]() -> int {
    FI_CUDA(cudaMemcpyAsync(d_blobs.get() + world, &mine, sizeof(mine), cudaMemcpyHostToDevice, h->s_main.get()));
    int rc = nccl_allgather(h, sh.comm.get(), d_blobs.get() + world, d_blobs.get(), sizeof(XchgBlob), h->s_main.get());
    if (rc != FI_OK) return rc;
    FI_CUDA(cudaMemcpyAsync(all.data(), d_blobs.get(), (size_t)world * sizeof(XchgBlob), cudaMemcpyDeviceToHost, h->s_main.get()));
    FI_CUDA(cudaStreamSynchronize(h->s_main.get()));
    return FI_OK;
  };
  int rc = gather();
  if (rc != FI_OK) return rc;
  bool ok = true;
  for (uint32_t k = 0; k < world; ++k) ok = ok && all[k].ok;
  if (ok) {
    for (uint32_t k = 0; k < world && ok; ++k) {
      if (k == rank) {
        px.base[k] = sh.d_xchg.get();
      } else if (all[k].pid == mine.pid) {  // same process: plain peer access
        int can = 0;
        if (all[k].device != h->cfg.device) {
          cudaDeviceCanAccessPeer(&can, h->cfg.device, all[k].device);
          if (can) {
            cudaError_t e = cudaDeviceEnablePeerAccess(all[k].device, 0);
            can = (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled);
            cudaGetLastError();
          }
        } else {
          can = 1;
        }
        ok = can != 0;
        px.base[k] = (uint8_t*)(uintptr_t)all[k].ptr;
      } else {
        void* m = nullptr;
        if (cudaIpcOpenMemHandle(&m, all[k].handle, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess) {
          sh.peer_ipc[k].reset(m);
          px.base[k] = (uint8_t*)m;
        } else {
          cudaGetLastError();
          ok = false;
        }
      }
    }
  }
  mine.ok = ok ? 1 : 0;
  rc = gather();
  if (rc != FI_OK) return rc;
  for (uint32_t k = 0; k < world; ++k) ok = ok && all[k].ok;
  if (ok) {
    px.enabled = 1;
    px.step = 0;
    *sh.h_xerr = 0;
    px.err = const_cast<uint32_t*>(sh.h_xerr.get());  // unified addressing: the host pointer is the device pointer
  }
  sh.px = px;
  if (std::getenv("FI_EPP_VERBOSE"))
    std::fprintf(stderr, "[fi_epp] rank %u/%u: sharded exchange over %s\n", rank, world,
                 px.enabled ? "peer memory (in-kernel tagged stores)" : "NCCL all-gather");
  return FI_OK;
}

// Build the shard of rank `rank` in a pool of `world` ranks: communicator, pick gather buffers, gossip logs and
// peer exchange.  On failure nothing of it survives.
int alloc_shard(fi_epp* h, const ncclUniqueId& id, uint32_t rank, uint32_t world, std::unique_ptr<Shard>* out) {
  auto sh = std::make_unique<Shard>();
  ncclComm_t comm = nullptr;
  int rc = g_nccl.CommInitRank(&comm, (int)world, id, (int)rank);
  if (rc != ncclSuccess)
    return fail(h, FI_ERR_COMM, std::string("ncclCommInitRank: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "error"));
  sh->comm.reset(comm);
  const uint64_t R = h->cfg.max_batch;
  FI_CUDA(dev_alloc(sh->d_local, R * h->P * sizeof(fi_pick)));
  FI_CUDA(dev_alloc(sh->d_gather, (size_t)world * R * h->P * sizeof(fi_pick)));
  // directory gossip (index_kernels.cu): this rank's transition log + gather buffers
  FI_CUDA(dev_alloc(sh->d_glog_n, 2 * sizeof(unsigned long long)));
  FI_CUDA(cudaMemset(sh->d_glog_n.get(), 0, 2 * sizeof(unsigned long long)));
  FI_CUDA(dev_alloc(sh->d_glog_a, kOpChunk * sizeof(uint64_t)));
  FI_CUDA(dev_alloc(sh->d_glog_v, kOpChunk * sizeof(uint64_t)));
  FI_CUDA(dev_alloc(sh->d_ghdr, (size_t)(world + 1) * 2 * sizeof(unsigned long long)));
  FI_CUDA(host_alloc(sh->h_ghdr, (size_t)(world + 1) * 2 * sizeof(unsigned long long)));
  FI_CUDA(dev_alloc(sh->d_ggather, (size_t)world * kOpChunk * sizeof(uint64_t)));
  rc = setup_peer_exchange(h, *sh, rank, world);
  if (rc != FI_OK) return rc;
  *out = std::move(sh);
  return FI_OK;
}

}  // namespace fi

int fi_epp_comm_unique_id(uint8_t out[FI_EPP_UNIQUE_ID_BYTES]) {
  if (!out) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(g_nccl_mu);
  std::string e;
  if (!g_nccl.load(&e)) {
    std::fprintf(stderr, "fi_epp_comm_unique_id: %s\n", e.c_str());
    return FI_ERR_COMM;
  }
  ncclUniqueId id;
  if (g_nccl.GetUniqueId(&id) != ncclSuccess) return FI_ERR_COMM;
  static_assert(sizeof(ncclUniqueId) == FI_EPP_UNIQUE_ID_BYTES, "unique id size");
  std::memcpy(out, &id, sizeof(id));
  return FI_OK;
}

int fi_epp_comm_init(fi_epp* h, const uint8_t id_bytes[FI_EPP_UNIQUE_ID_BYTES], uint32_t rank, uint32_t world) {
  if (!h || !id_bytes || world == 0 || rank >= world) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (h->shard) return fail(h, FI_ERR_STATE, "communicator already initialised");
  if (world > 32) return fail(h, FI_ERR_INVALID, "more than 32 ranks: the directory keeps one presence bit per rank");
  if (h->ops_applied || h->n_sets || h->n_clears)
    return fail(h, FI_ERR_STATE, "fi_epp_comm_init must precede the first index update (the directory is built by gossip)");
  if (world == 1) {
    h->rank = 0;
    h->world = 1;
    return FI_OK;
  }
  {
    std::lock_guard<std::mutex> lk2(g_nccl_mu);
    std::string e;
    if (!g_nccl.load(&e)) return fail(h, FI_ERR_COMM, e);
  }
  ncclUniqueId id;
  std::memcpy(&id, id_bytes, sizeof(id));
  int rc = alloc_shard(h, id, rank, world, &h->shard);  // (a failure leaves the handle a single rank)
  if (rc != FI_OK) return rc;
  h->rank = rank;
  h->world = world;
  return FI_OK;
}

int fi_epp_comm_exchange(fi_epp* h) {
  if (!h) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (h->world <= 1) return FI_EXCHANGE_NONE;
  return h->shard->px.enabled ? FI_EXCHANGE_PEER : FI_EXCHANGE_NCCL;
}
