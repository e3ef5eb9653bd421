// engine_index.cu — index ops: staging and flush, counters, rebuild, gossip rounds of sharded pools, host-LRU batch Add.
#include "engine.h"
#include <sched.h>

namespace fi {

// host cores this process may really use: the affinity mask capped by the cgroup CPU quota (more runnable
// threads than quota only get the group throttled)
unsigned usable_cores() {
  unsigned n = std::thread::hardware_concurrency();
  cpu_set_t set;
  CPU_ZERO(&set);
  if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) n = (unsigned)CPU_COUNT(&set);
  if (FILE* f = std::fopen("/sys/fs/cgroup/cpu.max", "r")) {  // cgroup v2: "<quota|max> <period>"
    char q[64] = {0};
    long long period = 0;
    if (std::fscanf(f, "%63s %lld", q, &period) == 2 && std::strcmp(q, "max") != 0 && period > 0) {
      const long long quota = std::atoll(q);
      if (quota > 0) n = std::min<unsigned>(n, (unsigned)std::max<long long>(1, (quota + period - 1) / period));
    }
    std::fclose(f);
  }
  return n ? n : 1u;
}

struct CopyJob {
  fi_index_op* dst;
  const fi_index_op* src;
  size_t n;
};

size_t index_bytes(uint64_t slots, uint32_t W) {
  const uint64_t total = slots + 3;
  return total * (sizeof(uint64_t) * 2 + sizeof(uint32_t) * 3 + (size_t)W * sizeof(uint32_t));
}

// queue the clears that make `v` an empty index (on the index stream)
int clear_index(fi_epp* h, const IndexView& v) {
  const uint64_t total = v.C + 3;
  FI_CUDA(cudaMemsetAsync(v.keys, 0, total * sizeof(uint64_t), h->s_index.get()));
  FI_CUDA(cudaMemsetAsync(v.node_of, 0xFF, total * sizeof(uint32_t), h->s_index.get()));  // NODE_INVALID
  FI_CUDA(cudaMemsetAsync(v.klog, 0, total * sizeof(uint64_t), h->s_index.get()));
  FI_CUDA(cudaMemsetAsync(v.rows, 0, total * v.W * sizeof(uint32_t), h->s_index.get()));
  FI_CUDA(cudaMemsetAsync(v.cnt, 0, total * sizeof(uint32_t), h->s_index.get()));
  FI_CUDA(cudaMemsetAsync(v.rmask, 0, total * sizeof(uint32_t), h->s_index.get()));
  return FI_OK;
}

int alloc_index(fi_epp* h, uint64_t slots, std::unique_ptr<IndexTable>* out) {
  auto t = std::make_unique<IndexTable>();
  IndexView& v = t->view;
  v.C = slots;
  v.bmask = slots / BUCKET_KEYS - 1;
  v.W = h->W;
  v.logW = 0;
  while ((1u << v.logW) < v.W) ++v.logW;
  const uint64_t total = slots + 3;  // + slots for hash 0, hash ~0, and a permanently-zero row
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && index_bytes(slots, v.W) + (256ull << 20) > free_b) {
    h->err = "index of " + std::to_string(index_bytes(slots, v.W) >> 20) + " MiB does not fit in the " +
             std::to_string(free_b >> 20) + " MiB of free device memory";
    return FI_ERR_NOMEM;
  }
  cudaError_t e = dev_alloc(t->keys, total * sizeof(uint64_t));
  if (e == cudaSuccess) e = dev_alloc(t->node_of, total * sizeof(uint32_t));
  if (e == cudaSuccess) e = dev_alloc(t->klog, total * sizeof(uint64_t));
  if (e == cudaSuccess) e = dev_alloc(t->rows, total * v.W * sizeof(uint32_t));
  if (e == cudaSuccess) e = dev_alloc(t->cnt, total * sizeof(uint32_t));
  if (e == cudaSuccess) e = dev_alloc(t->rmask, total * sizeof(uint32_t));
  if (e != cudaSuccess) {
    cudaGetLastError();
    h->err = std::string("index allocation: ") + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? FI_ERR_NOMEM : FI_ERR_CUDA;
  }
  v.keys = t->keys.get();
  v.node_of = t->node_of.get();
  v.klog = t->klog.get();
  v.rows = t->rows.get();
  v.cnt = t->cnt.get();
  v.rmask = t->rmask.get();
  int rc = clear_index(h, v);
  if (rc != FI_OK) return rc;
  *out = std::move(t);
  return FI_OK;
}

// Compact the live nodes into the spare table and swap.  Everything is queued on the index stream — no host
// synchronisation: picks submitted later wait for ev_index (recorded by the flush that called us) and are
// launched with the new view; picks already in flight keep reading the old tables, which are not touched again
// before the NEXT rebuild, and that one is ordered behind them (flush_ops makes s_index wait for ev_pick).
// The spare is allocated once, at the first rebuild (the only point where memory doubles), and then reused.
int rebuild_index(fi_epp* h) {
  int rc = h->ix_spare ? clear_index(h, h->ix_spare->view) : alloc_index(h, h->ix->view.C, &h->ix_spare);  // (alloc clears too)
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaMemsetAsync(h->d_ctr.get(), 0, sizeof(IndexCounters), h->s_index.get()));
  {
    LaunchScope ls(h, h->s_index.get(), K_INDEX);
    FI_CUDA(launch_index_rebuild(h->ix->view, h->ix_spare->view, h->d_ctr.get(), h->s_index.get()));
  }
  std::swap(h->ix, h->ix_spare);
  h->rebuilds++;
  return FI_OK;
}

// look at the counters copied back after the previous flush; rebuild if the table is
// clogged with tombstones, fail if it is genuinely full
int check_counters(fi_epp* h) {
  if (!h->ctr_pending) return FI_OK;
  FI_CUDA(cudaEventSynchronize(h->ev_ctr.get()));
  h->ctr_pending = false;
  if (h->dlru && h->dlru->stat->error)
    return fail(h, FI_ERR_STATE, "device LRU: invariant " + std::to_string(h->dlru->stat->error) + " broken");
  if (h->h_ctr->overflow) return fail(h, FI_ERR_CAPACITY, "index full: raise index_slots");
  const uint64_t used = h->h_ctr->used, tomb = h->h_ctr->tombstones;
  if (used * 10 > h->ix->view.C * 7) {
    if ((used - tomb) * 10 > h->ix->view.C * 6) return fail(h, FI_ERR_CAPACITY, "index above 60% live keys: raise index_slots");
    // the rebuild reads the old tables on s_index: every pick that still uses them must be ordered before the
    // NEXT rebuild clears them — flush_ops (our only caller that launches work) waits for ev_pick first
    FI_CUDA(cudaStreamWaitEvent(h->s_index.get(), h->ev_pick, 0));
    int rc = rebuild_index(h);
    if (rc != FI_OK) return rc;
    FI_CUDA(cudaEventRecord(h->ev_index.get(), h->s_index.get()));
  h->gen_index++;
  }
  return FI_OK;
}

GossipLog gossip_log(fi_epp* h) {
  GossipLog g{};
  if (h->shard) {
    g.n_appear = h->shard->d_glog_n.get();
    g.n_vanish = h->shard->d_glog_n.get() + 1;
    g.appear = h->shard->d_glog_a.get();
    g.vanish = h->shard->d_glog_v.get();
    g.cap = kOpChunk;
  }
  return g;
}

// launch the staged SET then CLEAR ops of the current group on the index stream.
// Asynchronous: the only waits are for the *previous* group's counters (rebuild /
// overflow decisions lag one group) and for the staging buffer being reused.
int flush_ops(fi_epp* h) {
  if (h->n_sets == 0 && h->n_clears == 0) return FI_OK;
  int rc = check_counters(h);  // may rebuild (swaps tables) — only ever between groups
  if (rc != FI_OK) return rc;
  const int b = h->cur_buf;
  // ops submitted after a pick returned must not overtake it on the GPU: the pick sees the index as of its call
  FI_CUDA(cudaStreamWaitEvent(h->s_index.get(), h->ev_pick, 0));
  const GossipLog gl = gossip_log(h);
  if (h->n_sets) {
    FI_CUDA(cudaMemcpyAsync(h->d_sets[b].get(), h->h_sets[b].get(), h->n_sets * sizeof(fi_index_op), cudaMemcpyHostToDevice, h->s_index.get()));
    h->stats.h2d_bytes += h->n_sets * sizeof(fi_index_op);
    LaunchScope ls(h, h->s_index.get(), K_INDEX);
    FI_CUDA(launch_index_set(h->ix->view, h->d_ctr.get(), h->d_sets[b].get(), h->n_sets, h->cfg.endpoint_begin, h->cfg.endpoint_count, h->rank,
                             gl, h->s_index.get()));
  }
  if (h->n_clears) {
    FI_CUDA(cudaMemcpyAsync(h->d_clears[b].get(), h->h_clears[b].get(), h->n_clears * sizeof(fi_index_op), cudaMemcpyHostToDevice, h->s_index.get()));
    h->stats.h2d_bytes += h->n_clears * sizeof(fi_index_op);
    LaunchScope ls(h, h->s_index.get(), K_INDEX);
    FI_CUDA(launch_index_clear(h->ix->view, h->d_ctr.get(), h->d_clears[b].get(), h->n_clears, h->cfg.endpoint_begin, h->cfg.endpoint_count,
                               h->rank, gl, h->s_index.get()));
  }
  h->ops_applied += h->n_sets + h->n_clears;
  FI_CUDA(cudaEventRecord(h->ev_buf[b].get(), h->s_index.get()));
  FI_CUDA(cudaMemcpyAsync(h->h_ctr.get(), h->d_ctr.get(), sizeof(IndexCounters), cudaMemcpyDeviceToHost, h->s_index.get()));
  FI_CUDA(cudaEventRecord(h->ev_ctr.get(), h->s_index.get()));
  h->ctr_pending = true;
  FI_CUDA(cudaEventRecord(h->ev_index.get(), h->s_index.get()));
  h->gen_index++;
  h->n_sets = h->n_clears = 0;
  h->cleared.clear();
  h->cur_buf ^= 1;
  // the buffer we are about to fill must have been consumed
  FI_CUDA(cudaEventSynchronize(h->ev_buf[h->cur_buf].get()));
  return FI_OK;
}

// Sharded pools, one gossip round (collective: every rank calls it the same number of times): exchange the
// transition logs written by this round's SET / CLEAR kernels and replay the other ranks' into the local
// directory — all APPEARs before all VANISHes, like the SETs and CLEARs that produced them.
int gossip_round(fi_epp* h) {
  if (h->world <= 1) return FI_OK;
  Shard& sh = *h->shard;
  const uint32_t Wd = h->world;
  int rc = nccl_allgather(h, sh.comm.get(), sh.d_glog_n.get(), sh.d_ghdr.get(), 2 * sizeof(unsigned long long), h->s_index.get());
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaMemcpyAsync(sh.h_ghdr.get(), sh.d_ghdr.get(), (size_t)Wd * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->s_index.get()));
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  const unsigned long long* hdr = sh.h_ghdr.get();
  uint64_t na = 0, nv = 0;
  for (uint32_t g = 0; g < Wd; ++g) {
    na = std::max<uint64_t>(na, hdr[2 * g]);
    nv = std::max<uint64_t>(nv, hdr[2 * g + 1]);
  }
  if (na > kOpChunk || nv > kOpChunk) return fail(h, FI_ERR_STATE, "gossip log overflow");
  if (na) {
    rc = nccl_allgather(h, sh.comm.get(), sh.d_glog_a.get(), sh.d_ggather.get(), na * sizeof(uint64_t), h->s_index.get());
    if (rc != FI_OK) return rc;
    for (uint32_t g = 0; g < Wd; ++g) {
      if (g == h->rank || hdr[2 * g] == 0) continue;
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_index_remote_appear(h->ix->view, h->d_ctr.get(), sh.d_ggather.get() + (size_t)g * na, hdr[2 * g], g, h->s_index.get()));
    }
  }
  if (nv) {
    rc = nccl_allgather(h, sh.comm.get(), sh.d_glog_v.get(), sh.d_ggather.get(), nv * sizeof(uint64_t), h->s_index.get());
    if (rc != FI_OK) return rc;
    for (uint32_t g = 0; g < Wd; ++g) {
      if (g == h->rank || hdr[2 * g + 1] == 0) continue;
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_index_remote_vanish(h->ix->view, h->d_ctr.get(), sh.d_ggather.get() + (size_t)g * nv, hdr[2 * g + 1], g, h->s_index.get()));
    }
  }
  FI_CUDA(cudaMemsetAsync(sh.d_glog_n.get(), 0, 2 * sizeof(unsigned long long), h->s_index.get()));
  if (na || nv) {  // the replays allocate nodes too: refresh the counters the rebuild decision reads
    FI_CUDA(cudaMemcpyAsync(h->h_ctr.get(), h->d_ctr.get(), sizeof(IndexCounters), cudaMemcpyDeviceToHost, h->s_index.get()));
    FI_CUDA(cudaEventRecord(h->ev_ctr.get(), h->s_index.get()));
    h->ctr_pending = true;
  }
  FI_CUDA(cudaEventRecord(h->ev_index.get(), h->s_index.get()));
  h->gen_index++;
  return FI_OK;
}

// Sharded pools: agree on how many gossip rounds a collective index call needs (the ranks' op counts differ)
int agree_rounds(fi_epp* h, uint64_t mine, uint64_t* rounds) {
  *rounds = mine;
  if (h->world <= 1) return FI_OK;
  Shard& sh = *h->shard;
  unsigned long long v[2] = {mine, 0};
  FI_CUDA(cudaMemcpyAsync(sh.d_ghdr.get() + 2 * (size_t)h->world, v, sizeof(v), cudaMemcpyHostToDevice, h->s_index.get()));
  int rc = nccl_allgather(h, sh.comm.get(), sh.d_ghdr.get() + 2 * (size_t)h->world, sh.d_ghdr.get(), sizeof(v), h->s_index.get());
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaMemcpyAsync(sh.h_ghdr.get(), sh.d_ghdr.get(), (size_t)h->world * sizeof(v), cudaMemcpyDeviceToHost, h->s_index.get()));
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  uint64_t m = 0;
  for (uint32_t g = 0; g < h->world; ++g) m = std::max<uint64_t>(m, sh.h_ghdr.get()[2 * g]);
  *rounds = m;
  return FI_OK;
}

// stage one op (already filtered to this shard).  Within a launch group SETs run
// before CLEARs, so a SET that follows a CLEAR of the same pair starts a new group.
int submit_op(fi_epp* h, uint64_t hash, uint32_t endpoint, uint32_t op) {
  if (op == FI_OP_SET) {
    if (!h->cleared.empty() && h->cleared.count(PairKey{hash, endpoint})) {
      int rc = flush_ops(h);
      if (rc != FI_OK) return rc;
    }
    h->h_sets[h->cur_buf].get()[h->n_sets++] = fi_index_op{hash, endpoint, FI_OP_SET};
  } else {
    h->cleared.insert(PairKey{hash, endpoint});
    h->h_clears[h->cur_buf].get()[h->n_clears++] = fi_index_op{hash, endpoint, FI_OP_CLEAR};
  }
  if (h->n_sets == kOpChunk || h->n_clears == kOpChunk) return flush_ops(h);
  return FI_OK;
}

}  // namespace fi

// One collective index update of a sharded pool = `rounds` gossip rounds on every rank; `step(i)` stages and
// flushes this rank's share of round i (nothing if it has fewer).  Single rank: just the steps.
static int run_rounds(fi_epp* h, uint64_t mine, int my_err, const std::function<int(uint64_t)>& step) {
  if (h->world <= 1) {
    if (my_err != FI_OK) return my_err;
    for (uint64_t i = 0; i < mine; ++i) {
      int rc = step(i);
      if (rc != FI_OK) return rc;
    }
    return FI_OK;
  }
  // a rank whose arguments were rejected still takes part (with zero rounds) so that the others do not hang
  uint64_t rounds = 0;
  int rc = agree_rounds(h, my_err == FI_OK ? mine : 0, &rounds);
  if (rc != FI_OK) return rc;
  for (uint64_t i = 0; i < rounds; ++i) {
    if (my_err == FI_OK && i < mine) {
      rc = step(i);
      if (rc != FI_OK) return rc;
    }
    rc = gossip_round(h);
    if (rc != FI_OK) return rc;
  }
  return my_err;
}

int fi_epp_index_apply(fi_epp* h, const fi_index_op* ops, uint64_t n) {
  if (!h || (!ops && n)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  int err = check_counters(h);
  for (uint64_t i = 0; i < n && err == FI_OK; ++i) {
    if (ops[i].op != FI_OP_SET && ops[i].op != FI_OP_CLEAR) err = fail(h, FI_ERR_INVALID, "bad index opcode");
    else if (ops[i].endpoint >= h->cfg.num_endpoints) err = fail(h, FI_ERR_INVALID, "index op endpoint out of range");
  }
  const uint32_t lo = h->cfg.endpoint_begin, cnt = h->cfg.endpoint_count;
  // rounds of kOpChunk input ops: a round never overflows the staging buffers (or, sharded, the gossip log)
  const uint64_t rounds = (n + kOpChunk - 1) / kOpChunk;
  return run_rounds(h, rounds, err, [&](uint64_t i) -> int {
    const uint64_t i0 = i * kOpChunk, i1 = std::min(n, i0 + kOpChunk);
    for (uint64_t k = i0; k < i1; ++k) {
      const fi_index_op& op = ops[k];
      if (op.endpoint - lo >= cnt) continue;  // another rank's shard
      int rc = submit_op(h, op.hash, op.endpoint, op.op);
      if (rc != FI_OK) return rc;
    }
    return flush_ops(h);
  });
}

int fi_epp_index_add_chain(fi_epp* h, uint32_t endpoint, const uint64_t* hashes, uint32_t n) {
  if (!h || (!hashes && n)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (!h->cfg.lru_capacity) return fail(h, FI_ERR_STATE, "lru_capacity is 0: the host LRU is disabled");
  if (h->world > 1) return fail(h, FI_ERR_STATE, "sharded pool: use the collective fi_epp_index_add_chains");  // (device LRU too)
  if (endpoint >= h->cfg.num_endpoints) return fail(h, FI_ERR_INVALID, "endpoint out of range");
  const uint32_t e = endpoint - h->cfg.endpoint_begin;
  if (e >= h->cfg.endpoint_count) return FI_OK;  // another rank's shard
  int rc = choose_lru_mode(h);
  if (rc != FI_OK) return rc;
  if (h->lru_mode == 1) return lru_device_add(h, &endpoint, hashes, false, n, &n, 1);
  rc = check_counters(h);
  if (rc != FI_OK) return rc;
  LruSet& l = h->lrus[e];
  for (uint32_t i = 0; i < n; ++i) {
    uint64_t ev = 0;
    bool did = false;
    const bool inserted = l.touch(hashes[i], &ev, &did);
    if (did) {
      rc = submit_op(h, ev, endpoint, FI_OP_CLEAR);
      if (rc != FI_OK) return rc;
    }
    if (inserted) {
      rc = submit_op(h, hashes[i], endpoint, FI_OP_SET);
      if (rc != FI_OK) return rc;
    }
  }
  // the deltas stay staged: they are launched when the staging buffer fills and, at the latest,
  // by the next pick / sync (one launch group per batch of decisions instead of one per chain)
  return FI_OK;
}

// Upstream PreRequest for a whole batch of decisions: indexer.Add(chain_r, endpoints[r]) for r = 0..R-1, in
// request order per endpoint (the endpoints' LRUs are independent of each other, so they are walked in
// parallel on the host worker pool; the result equals R sequential fi_epp_index_add_chain calls).
int fi_epp_index_add_chains(fi_epp* h, const uint32_t* endpoints, const uint64_t* chains, uint32_t pitch_blocks,
                            const uint32_t* nblocks, uint32_t R) {
  if (!h || ((!endpoints || !chains || !nblocks) && R)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  int err = FI_OK;
  if (!h->cfg.lru_capacity) err = fail(h, FI_ERR_STATE, "lru_capacity is 0: the host LRU is disabled");
  for (uint32_t r = 0; r < R && err == FI_OK; ++r) {
    if (endpoints[r] != FI_NO_ENDPOINT && endpoints[r] >= h->cfg.num_endpoints) err = fail(h, FI_ERR_INVALID, "endpoint out of range");
    else if (nblocks[r] > pitch_blocks) err = fail(h, FI_ERR_INVALID, "nblocks[r] larger than the chain pitch");
  }
  if (err == FI_OK) err = choose_lru_mode(h);
  if (err == FI_OK && h->lru_mode == 1) return lru_device_add(h, endpoints, chains, false, pitch_blocks, nblocks, R);
  if (err == FI_OK) err = check_counters(h);

  // ---- 1./2. bucket the requests by endpoint and walk the LRUs on the worker pool (lru_batch.h)
  const uint32_t lo = h->cfg.endpoint_begin, EL = h->cfg.endpoint_count;
  std::vector<WorkerOps>& outs = h->lru_outs;  // persistent: capacity survives from batch to batch
  size_t nseg = 0;
  const auto t_start = std::chrono::steady_clock::now();
  if (!h->pool) {
    unsigned t = std::min(usable_cores(), 128u);
    if (const char* ev = std::getenv("FI_EPP_LRU_THREADS")) t = (unsigned)std::max(1L, std::strtol(ev, nullptr, 10));
    if (h->lru_threads) t = h->lru_threads;
    h->pool.reset(new WorkerPool(t));
  }
  if (err == FI_OK) nseg = lru_walk_batch(h->lrus, lo, EL, endpoints, chains, pitch_blocks, nblocks, R, *h->pool, outs);
  else for (auto& o : outs) o.begin_batch();
  const auto t_walked = std::chrono::steady_clock::now();

  // ---- 3. stage segment by segment (SETs, then CLEARs), flushing whenever a staging buffer is full.
  // `flushes` is first counted (dry run) so that the ranks of a sharded pool can agree on the rounds.
  std::vector<CopyJob> jobs;
  auto run_jobs = [&]() {
    if (jobs.empty()) return;
    // big copies into the pinned staging buffers go through the worker pool
    std::vector<CopyJob> pieces;
    const size_t kPiece = 1u << 16;
    for (const CopyJob& j : jobs)
      for (size_t o = 0; o < j.n; o += kPiece) pieces.push_back(CopyJob{j.dst + o, j.src + o, std::min(kPiece, j.n - o)});
    h->pool->run((uint32_t)pieces.size(), [&](uint32_t t, unsigned) {
      std::memcpy(pieces[t].dst, pieces[t].src, pieces[t].n * sizeof(fi_index_op));
    });
    jobs.clear();
  };
  // walk(dry): returns the number of flushes; !dry performs them through do_flush
  auto walk = [&](bool dry, const std::function<int()>& do_flush, uint64_t* n_flush) -> int {
    uint64_t ns = dry ? 0 : h->n_sets, nc = dry ? 0 : h->n_clears, flushes = 0;
    auto flush = [&]() -> int {
      ++flushes;
      if (!dry) {
        run_jobs();
        h->n_sets = ns;
        h->n_clears = nc;
        int rc = do_flush();
        if (rc != FI_OK) return rc;
      }
      ns = nc = 0;
      return FI_OK;
    };
    for (size_t seg = 0; seg < nseg; ++seg) {
      for (int kind = 0; kind < 2; ++kind) {
        for (auto& o : outs) {
          if (o.nseg <= seg) continue;
          const std::vector<fi_index_op>& v = kind == 0 ? o.sets[seg] : o.clears[seg];
          size_t done = 0;
          while (done < v.size()) {
            uint64_t& fillc = kind == 0 ? ns : nc;
            const size_t room = (size_t)(kOpChunk - fillc);
            const size_t take = std::min(room, v.size() - done);
            if (!dry && take) {
              fi_index_op* base = kind == 0 ? h->h_sets[h->cur_buf].get() : h->h_clears[h->cur_buf].get();
              jobs.push_back(CopyJob{base + fillc, v.data() + done, take});
            }
            fillc += take;
            done += take;
            if (fillc == kOpChunk) {
              int rc = flush();
              if (rc != FI_OK) return rc;
            }
          }
        }
      }
      if (seg + 1 < nseg && (ns || nc)) {  // segment boundary: the next segment's SETs must run after these CLEARs
        int rc = flush();
        if (rc != FI_OK) return rc;
      }
    }
    if (!dry) {
      run_jobs();
      h->n_sets = ns;
      h->n_clears = nc;
    }
    if (n_flush) *n_flush = flushes;
    return FI_OK;
  };

  if (h->world <= 1) {
    if (err != FI_OK) return err;
    // the tail stays staged: it is launched with the next flush — at the latest by the next pick / sync
    int rc1 = walk(false, [&]() { return flush_ops(h); }, nullptr);
    if (h->verbose) {
      const auto t_end = std::chrono::steady_clock::now();
      size_t nops = 0;
      for (auto& o : outs)
        for (size_t sg = 0; sg < o.nseg; ++sg) nops += o.sets[sg].size() + o.clears[sg].size();
      std::fprintf(stderr, "[fi_epp] add_chains: %u requests, %zu ops, %zu segment(s), %u workers: LRU walk %.2f ms, staging %.2f ms\n",
                   R, nops, nseg, h->pool->size(), std::chrono::duration<double, std::milli>(t_walked - t_start).count(),
                   std::chrono::duration<double, std::milli>(t_end - t_walked).count());
    }
    return rc1;
  }
  // sharded: every flush is one gossip round, the tail included
  uint64_t mine = 0;
  if (err == FI_OK) {
    walk(true, nullptr, &mine);
    mine += 1;  // the tail
  }
  uint64_t rounds = 0;
  int rc = agree_rounds(h, err == FI_OK ? mine : 0, &rounds);
  if (rc != FI_OK) return rc;
  uint64_t did = 0;
  if (err == FI_OK) {
    rc = walk(false, [&]() -> int {
      int r2 = flush_ops(h);
      if (r2 != FI_OK) return r2;
      ++did;
      return gossip_round(h);
    }, nullptr);
    if (rc != FI_OK) return rc;
    rc = flush_ops(h);  // the tail
    if (rc != FI_OK) return rc;
  }
  for (; did < rounds; ++did) {
    rc = gossip_round(h);
    if (rc != FI_OK) return rc;
  }
  return err;
}

int fi_epp_index_sync(fi_epp* h) {
  if (!h) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  int rc = flush_ops(h);
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  return check_counters(h);
}

int fi_epp_index_stats(fi_epp* h, fi_index_stats* out) {
  if (!h || !out) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  int rc = flush_ops(h);
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  IndexCounters c;
  FI_CUDA(cudaMemcpy(&c, h->d_ctr.get(), sizeof(c), cudaMemcpyDeviceToHost));
  out->slots = h->ix->view.C;
  out->used = c.used;
  out->tombstones = c.tombstones;
  out->rebuilds = h->rebuilds;
  out->ops_applied = h->ops_applied;
  uint64_t l = 0;
  if (h->lru_mode == 1 && h->dlru) {
    std::vector<uint32_t> cnt(h->dlru->view.EL);
    FI_CUDA(cudaMemcpy(cnt.data(), h->dlru->view.count, cnt.size() * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (uint32_t c2 : cnt) l += c2;
    out->ops_applied += h->dlru->stat->n_sets + h->dlru->stat->n_clears;
  } else {
    for (auto& s : h->lrus) l += s.size();
  }
  out->lru_entries = l;
  return FI_OK;
}

// diagnostics for tests: out[i] = 1 iff (ops[i].endpoint, ops[i].hash) is in the GPU index
int fi_epp_index_contains(fi_epp* h, const fi_index_op* q, uint64_t n, uint8_t* out) {
  if (!h || (!q && n) || (!out && n)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  int rc = flush_ops(h);
  if (rc != FI_OK) return rc;
  if (n == 0) return FI_OK;
  DevPtr<fi_index_op> dq;
  DevPtr<uint8_t> dout;
  FI_CUDA(dev_alloc(dq, n * sizeof(fi_index_op)));
  if (dev_alloc(dout, n) != cudaSuccess) return fail(h, FI_ERR_NOMEM, "cudaMalloc failed");
  FI_CUDA(cudaMemcpyAsync(dq.get(), q, n * sizeof(fi_index_op), cudaMemcpyHostToDevice, h->s_index.get()));
  {
    LaunchScope ls(h, h->s_index.get(), K_OTHER);
    FI_CUDA(launch_index_contains(h->ix->view, dq.get(), n, h->cfg.endpoint_begin, h->cfg.endpoint_count, dout.get(), h->s_index.get()));
  }
  FI_CUDA(cudaMemcpyAsync(out, dout.get(), n, cudaMemcpyDeviceToHost, h->s_index.get()));
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  return FI_OK;
}
