// engine.h — private header of the host side of libfi_epp (engine*.cu): the handle and its parts, the owners of
// their CUDA resources.  The handle owns the device buffers, two CUDA streams (compute, index maintenance), the
// pinned op ring that keeps the GPU index live (async H2D on the side stream, ordered before the next pick), the
// host LRU, the per-batch score tables, and the optional NCCL communicator for endpoint-range sharded pools.
// The entry points of include/fi_epp.h take their C linkage from that header.  No CPU fallback: creation fails
// without a CUDA device.
#pragma once
#include <cuda.h>  // types and prototypes of the green-context API only: reached through cudaGetDriverEntryPoint, libcuda is not linked
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <type_traits>
#include <unordered_set>
#include <vector>

#include "../../include/fi_epp.h"
#include "kernels.cuh"
#include "lru.h"
#include "lru_batch.h"
#include "lru_device.cuh"
#include "lru_plan.h"
#include "xxh64.cuh"

using namespace fi;

typedef struct ncclComm* ncclComm_t;

namespace fi {

// ---- owners of the handle's CUDA resources: move-only, each releases its resource when it goes away ----
void green_ctx_destroy(CUgreenCtx c);  // through the driver entry point (g_green)
void comm_destroy(ncclComm_t c);       // through the dlopen'ed NCCL (g_nccl)
template <auto Release>
struct Releaser {
  template <typename T>
  void operator()(T* p) const { Release(const_cast<std::remove_cv_t<T>*>(p)); }
};
template <typename T>
using DevPtr = std::unique_ptr<T, Releaser<cudaFree>>;  // cudaMalloc
template <typename T>
using HostPtr = std::unique_ptr<T, Releaser<cudaFreeHost>>;  // pinned: cudaHostAlloc
using Event = std::unique_ptr<CUevent_st, Releaser<cudaEventDestroy>>;
using Stream = std::unique_ptr<CUstream_st, Releaser<cudaStreamDestroy>>;  // runtime streams and those of green contexts
using GreenCtx = std::unique_ptr<CUgreenCtx_st, Releaser<green_ctx_destroy>>;
using NcclComm = std::unique_ptr<ncclComm, Releaser<comm_destroy>>;
using IpcMapping = std::unique_ptr<void, Releaser<cudaIpcCloseMemHandle>>;  // cudaIpcOpenMemHandle

// (the previous resource is released first: a buffer that grows never holds both sizes)
template <typename T>
cudaError_t dev_alloc(DevPtr<T>& p, size_t bytes) {
  p.reset();
  void* q = nullptr;
  const cudaError_t e = cudaMalloc(&q, bytes);
  p.reset(e == cudaSuccess ? static_cast<T*>(q) : nullptr);
  return e;
}
template <typename T>
cudaError_t host_alloc(HostPtr<T>& p, size_t bytes, unsigned flags = cudaHostAllocDefault) {
  p.reset();
  void* q = nullptr;
  const cudaError_t e = cudaHostAlloc(&q, bytes, flags);
  p.reset(e == cudaSuccess ? static_cast<T*>(q) : nullptr);
  return e;
}
inline cudaError_t event_create(Event& ev, unsigned flags = cudaEventDisableTiming) {
  cudaEvent_t e = nullptr;
  const cudaError_t r = cudaEventCreateWithFlags(&e, flags);
  ev.reset(r == cudaSuccess ? e : nullptr);
  return r;
}

struct PairKey {
  uint64_t hash;
  uint32_t endpoint;
  bool operator==(const PairKey& o) const { return hash == o.hash && endpoint == o.endpoint; }
};
struct PairHash {
  size_t operator()(const PairKey& k) const {
    uint64_t x = k.hash ^ ((uint64_t)k.endpoint * 0x9E3779B97F4A7C15ULL);
    x ^= x >> 29;
    return (size_t)(x * 0xBF58476D1CE4E5B9ULL);
  }
};

constexpr uint64_t kOpChunk = 1ull << 20;  // ops per pinned staging buffer

inline uint32_t pow2_ceil32(uint32_t v) {
  uint32_t p = 1;
  while (p < v) p <<= 1;
  return p;
}
inline uint64_t pow2_ceil64(uint64_t v) {
  uint64_t p = 1;
  while (p < v) p <<= 1;
  return p;
}

enum KernelKind { K_HASH = 0, K_CHAIN = 1, K_MATCH = 2, K_INDEX = 3, K_OTHER = 4, K_KINDS = 5 };

// ---- the parts of the handle.  A part created after fi_epp_create is built by one function that either hands
// over a complete part or leaves nothing behind; the handle holds it as a unique_ptr (null: not there).
// Members are released in the reverse order of their declaration.

// GPU index: the view the kernels take, filled from its owners
struct IndexTable {
  IndexView view{};
  DevPtr<uint64_t> keys, klog;
  DevPtr<uint32_t> node_of, rows, cnt, rmask;
};

// device-resident LRU (lru_kernels.cu): allocated at the first Add
struct DeviceLru {
  struct HostStat {
    uint32_t error, any_ovf;  // (any_ovf: the touch kernel's overflow flag of the running sub-batch)
    unsigned long long n_sets, n_maintained, n_clears_cur, n_clears, n_doomed;
  };
  DevLru view{};
  DevPtr<LruSlot> slots;
  DevPtr<uint64_t> log;
  DevPtr<uint32_t> state;               // head | tail | count | used | error
  DevPtr<unsigned long long> ctr;       // [0] SETs emitted, [1] endpoints maintained, [2] CLEARs of the running sub-batch,
                                        // [3] CLEARs total, [4] doomed winners
  HostPtr<HostStat> stat;               // pinned copy, refreshed after every call
  DevPtr<uint32_t> slot_of, wcount, base;
  DevPtr<fi_index_op> sets, clears;
  uint64_t touch_cap = 0;               // touches per sub-batch the scratch arrays hold
  DevPtr<uint32_t> d_plan;              // the planner's arrays of the current call
  HostPtr<uint32_t> h_plan;             // pinned staging of the same
  size_t plan_cap = 0;                  // in u32 words
  DevPtr<uint64_t> chains;              // staging of host chains
  size_t chains_cap = 0;                // in u64 words
  Event ev;                             // the previous call's staging has been consumed
  Event ev_ovf;                         // the touch kernel's overflow flag has reached the host
};

// second buffer slot of the pipelined path: allocated at the first fi_epp_pick_submit
struct PipeSlot {
  DevPtr<uint64_t> chain;
  DevPtr<uint32_t> nblocks;
};

// SM partition of the pipelined path (green contexts): built at the first submit or by the option "pipe_partition"
struct Partition {
  GreenCtx gctx_walk, gctx_main;  // (declared before their streams: released after them)
  Stream s_pw, s_pa, s_pb;        // walker | hashing, matching (big partition)
  DevPtr<uint64_t> d_pre2;
  DevPtr<uint32_t> d_nblocks3;
  Event ev_h[2], ev_b3[3], ev_up;
  int walk_sms = 0, main_sms = 0;
};

// endpoint-range sharded pool: built by fi_epp_comm_init
struct Shard {
  DevPtr<fi_pick> d_local;   // [R][P] this rank's picks
  DevPtr<fi_pick> d_gather;  // [world][R][P]
  // directory gossip (index_kernels.cu): this rank's transition log of the current round and the buffers the ranks'
  // logs are gathered into
  DevPtr<unsigned long long> d_glog_n;  // [2] appear / vanish counts
  DevPtr<uint64_t> d_glog_a, d_glog_v;  // [kOpChunk] each
  DevPtr<unsigned long long> d_ghdr;    // [world][2] gathered counts
  HostPtr<unsigned long long> h_ghdr;   // pinned copy
  DevPtr<uint64_t> d_ggather;           // [world][kOpChunk]
  // peer-memory exchange (kernels.cuh PeerXchg)
  PeerXchg px{};                        // px.enabled == 0: NCCL all-gathers are used
  DevPtr<uint8_t> d_xchg;               // this rank's exchange buffer
  HostPtr<volatile uint32_t> h_xerr;    // poll-timeout flag of the exchange (mapped pinned host word the kernels set)
  IpcMapping peer_ipc[FI_MAX_RANKS];    // the peers' buffers (closed before d_xchg is freed)
  NcclComm comm;                        // (declared last: destroyed first)
};

}  // namespace fi

struct fi_epp {
  fi_epp_config cfg;
  std::mutex mu;
  std::string err;
  int sm_count = 148;
  uint32_t MP = 0;  // chain pitch
  uint32_t W = 0;   // words per index row
  uint32_t P = 0;   // profiles
  bool fast_hash = false;

  // (the streams are declared first: every other resource of the handle is released before them)
  Stream s_main, s_index;  // compute; index maintenance (side stream)
  // host-buffer picks feed the prompts in slices: the copy engine runs ahead on s_copy while s_main hashes,
  // walks and matches the slices that have landed (the step is PCIe-bound: only the last slice's work is exposed)
  Stream s_copy;
  static constexpr int kMaxFeedSlices = 16;
  Event ev_copy[kMaxFeedSlices];
  uint32_t feed_slices = 8;  // FI_EPP_FEED_SLICES (1: one copy, then the whole batch)
  // Pipelined device path (fi_epp_pick_submit / fi_epp_pick_wait): stage A (block hashing + chain walk) of
  // batch k+1 runs on s_a while stage B (match + pick) of batch k runs on s_main; the chain / block-count
  // buffers are double-buffered (slot = batch parity: d_chain / d_nblocks and slot2), the pre-states are not
  // (stage A is serial on s_a).
  Stream s_a;
  std::unique_ptr<PipeSlot> slot2;
  Event ev_in, ev_a[2], ev_b[2];
  cudaEvent_t ev_pick = nullptr;  // completion of the most recent pick of any kind: ev_pick_own, or (partitioned
                                  // pipeline) the slot event of the batch submitted last — a handle, not a second record
  Event ev_pick_own;
  Event ev_plain;  // completion of the most recent stream-ordered (not pipelined) pick
  uint64_t pipe_seq = 0;          // batches submitted
  uint32_t pipe_hash_ctas = 0;    // per-SM caps of the pipelined path's two co-running kernels (0 = uncapped);
  uint32_t pipe_match_ctas = 0;   // FI_EPP_PIPE_HASH_CTAS / FI_EPP_PIPE_MATCH_CTAS, option "pipe_hash_ctas" / "pipe_match_ctas"
  // SM-partitioned pipeline (green contexts, CUDA 12.4+): the chain walk is serial latency that fills 6 % of the
  // warp slots but cannot share schedulers with a busy kernel (it slows 3x), so nothing overlapped it and every
  // batch paid its 27 us.  With the GPU split into a 40-SM partition for the walker (three or four of its warps per
  // scheduler) and a 108-SM partition for hash_blocks / match_pick, batch k is matched while batch k+1's chains
  // are walked and batch k+2 is hashed: three batches in flight, 131 -> 116 us per batch.
  // FI_EPP_PIPE_PARTITION=<SMs> / option "pipe_partition" (0 = off: two batches in flight on the whole GPU).
  // SMs asked for the walker partition.  Measured at cfg 3 (us per step; no partition: 131.1): 8 -> 240, 16 -> 125.6,
  // 24 -> 123.0, 32 -> 129.0, 40 -> 116.2 (three runs), 48 -> 124.3, 56 -> 133.7
  int part_want = 40;
  int part_compact = -1;        // walker shape on the partition: -1 = the 64-register shape only where the 78-register one does
                                // not fit (fewer than 24 SMs); FI_EPP_WALK_COMPACT=0/1 forces it
  bool part_tried = false;      // setup_partition has run since part_want was last set
  std::unique_ptr<Partition> part;  // null: not tried yet or unavailable (fallback to the unpartitioned pipeline)
  bool part_active = false;     // the partitioned pipeline has batches in flight / owns the slot events
  // how often ev_index / ev_plain / ev_lru have been re-recorded, and the values the partitioned pipeline's streams
  // already waited for: a submit makes ~16 runtime calls instead of ~23 (eight processes on a 16-core host are
  // launch-bound otherwise)
  uint64_t gen_index = 0, gen_plain = 0, gen_lru = 0;
  uint64_t seen_index = ~0ull, seen_plain = ~0ull, seen_lru = ~0ull;
  uint64_t part_seq = 0;        // batches submitted to it since it last became active
  Event ev_index, ev_user, ev_done, ev_ctr;

  // request buffers (device)
  DevPtr<uint8_t> d_prompts;
  DevPtr<uint64_t> d_offsets, d_h0, d_pre, d_chain;
  DevPtr<uint32_t> d_nblocks;
  DevPtr<fi_pick> d_picks;   // [R][P] final
  // sharded mode: every rank hashes every prompt (the default: 149 vs 141 M decisions/s at cfg 4 on 8 GPUs, 131 vs
  // 119 on 2 — hashing 16 KiB from local HBM costs less than receiving 2 KiB of chain over NVLink); FI_EPP_SHARD_HASH=
  // split / option "shard_hash" = 1: every rank hashes R/world requests and the chains are all-gathered
  bool split_hash = false;
  uint32_t chain_rows = 0;  // rows allocated in d_chain / d_pre / d_nblocks (max_batch padded for the gather)
  DevPtr<unsigned long long> d_probed;
  DevPtr<uint32_t> d_work;  // [16] dynamic work-queue counters of in-flight match launches
  // pinned host mirrors
  HostPtr<fi_pick> h_picks;
  HostPtr<uint64_t> h_offsets, h_h0;
  HostPtr<uint32_t> h_nblocks;

  // index
  std::unique_ptr<IndexTable> ix, ix_spare;  // ix_spare: rebuild target, allocated at the first rebuild and reused alternately
  DevPtr<IndexCounters> d_ctr;
  HostPtr<IndexCounters> h_ctr;  // pinned
  bool ctr_pending = false;
  uint64_t rebuilds = 0, ops_applied = 0;
  HostPtr<fi_index_op> h_sets[2], h_clears[2];
  DevPtr<fi_index_op> d_sets[2], d_clears[2];
  Event ev_buf[2];
  int cur_buf = 0;
  uint64_t n_sets = 0, n_clears = 0;
  std::unordered_set<PairKey, PairHash> cleared;
  LruArena lru_arena;  // backing store of the LRUs (one huge-page mapping)
  std::vector<LruSet> lrus;
  std::unique_ptr<WorkerPool> pool;  // host LRU workers (fi_epp_index_add_chains), created on first use
  std::vector<WorkerOps> lru_outs;   // their op lists (capacity kept from batch to batch)
  bool verbose = false;              // FI_EPP_VERBOSE
  // device-resident LRU (lru_kernels.cu): the default for single-rank handles whose lru_capacity holds a whole
  // chain; option "device_lru" / FI_EPP_DEVICE_LRU=0 selects the host LRU instead.  Allocated at the first Add;
  // the two are never mixed on one handle.
  int lru_mode = -1;  // -1: not chosen yet, 0: host LRU, 1: device LRU
  int lru_want = -1;  // option / environment override (-1: automatic)
  uint32_t lru_table_slots = 0;  // option "lru_table_slots": slots per endpoint table of the device LRU (0: sized by free HBM)
  std::unique_ptr<DeviceLru> dlru;
  uint64_t lru_deferred = 0, lru_sub_batches = 0;  // host-side totals
  uint32_t last_plain_R = 0;                 // rows of d_chain the most recent stream-ordered pick wrote
  LruPlan lru_plan;
  unsigned lru_threads = 0;          // 0: FI_EPP_LRU_THREADS, else min(usable cores, 64)

  // endpoints / score tables
  std::vector<EndpointDev> eps;  // global pool
  bool eps_dirty = true;
  DevPtr<EndpointDev> d_eps;
  DevPtr<double> d_sc;
  DevPtr<uint32_t> d_elig;
  DevPtr<ZeroBest> d_zero;
  DevPtr<uint32_t> d_ztie;
  std::vector<LoraDev> lora;   // local endpoints' adapter residency (lora-affinity-scorer)
  bool lora_dirty = false;
  DevPtr<LoraDev> d_lora;
  DevPtr<uint64_t> d_adapters;  // staging of the host path's per-request adapter ids
  HostPtr<uint64_t> h_adapters;  // pinned
  ScoreTables st{};

  // multi-GPU
  std::unique_ptr<Shard> shard;  // null: a single rank (world == 1)
  uint32_t rank = 0, world = 1;

  // stats / profiling
  fi_epp_stats stats{};
  bool profiling = false;
  bool tracing = false;       // FI_EPP_TRACE=<call index>: print that call's kernel timeline to stderr
  long trace_call = -1;
  Event ev_trace0;
  std::vector<Event> ev_pool;
  struct Ev {
    Event a, b;
    int kind;
  };
  std::vector<Ev> pending_ev;  // (declared after the pool: fi_epp_destroy drains it into the pool first)
};

namespace fi {

#define FI_CUDA(call)                                                                   \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e__);                     \
      return FI_ERR_CUDA;                                                               \
    }                                                                                   \
  } while (0)

inline int fail(fi_epp* h, int code, const std::string& m) {
  h->err = m;
  return code;
}

// an event for a profiled launch: from the pool, or a new one (null if that fails: the launch goes unprofiled)
inline Event get_event(fi_epp* h) {
  Event e;
  if (!h->ev_pool.empty()) {
    e = std::move(h->ev_pool.back());
    h->ev_pool.pop_back();
  } else {
    event_create(e, cudaEventDefault);
  }
  return e;
}

// wraps one kernel launch: counts it and, when profiling, brackets it with events
struct LaunchScope {
  fi_epp* h;
  cudaStream_t s;
  int kind;
  Event a, b;
  LaunchScope(fi_epp* h_, cudaStream_t s_, int kind_) : h(h_), s(s_), kind(kind_) {
    h->stats.kernel_launches++;
    if (h->profiling || h->tracing) {
      a = get_event(h);
      b = get_event(h);
      if (a && b) cudaEventRecord(a.get(), s);
    }
  }
  ~LaunchScope() {
    if (a && b) {
      cudaEventRecord(b.get(), s);
      h->pending_ev.push_back({std::move(a), std::move(b), kind});
    }
  }
};

// engine_index.cu
int alloc_index(fi_epp* h, uint64_t slots, std::unique_ptr<IndexTable>* out);
int check_counters(fi_epp* h);
int flush_ops(fi_epp* h);
GossipLog gossip_log(fi_epp* h);
int gossip_round(fi_epp* h);
int agree_rounds(fi_epp* h, uint64_t mine, uint64_t* rounds);
// engine_lru.cu
int choose_lru_mode(fi_epp* h);
int lru_device_add(fi_epp* h, const uint32_t* endpoints, const uint64_t* chains, bool on_device, uint32_t pitch,
                   const uint32_t* nblocks, uint32_t R, bool conservative = false);
// engine_comm.cu
int nccl_allgather(fi_epp* h, ncclComm_t comm, const void* send, void* recv, size_t bytes, cudaStream_t s);

}  // namespace fi
