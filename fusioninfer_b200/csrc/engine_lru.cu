// engine_lru.cu — device-resident LRU (lru_kernels.cu): Add, dump, counters.
#include "engine.h"

namespace fi {

// Which LRU serves this handle's indexer.Add calls: decided at the first one.
int choose_lru_mode(fi_epp* h) {
  if (h->lru_mode >= 0) return FI_OK;
  int want = h->lru_want;
  if (want < 0) {
    if (const char* e = std::getenv("FI_EPP_DEVICE_LRU")) want = std::strtol(e, nullptr, 10) != 0;
  }
  const bool possible = h->cfg.lru_capacity >= h->cfg.max_blocks && h->cfg.lru_capacity <= (1u << 28);
  if (want == 1 && !possible) return fail(h, FI_ERR_STATE, "device_lru needs lru_capacity >= max_blocks");
  h->lru_mode = (want < 0 ? possible : want == 1) ? 1 : 0;
  return FI_OK;
}

// Build the device LRU; on failure nothing of it survives (a later call may succeed, e.g. with the host LRU freed).
int alloc_dev_lru(fi_epp* h, std::unique_ptr<DeviceLru>* out) {
  auto L = std::make_unique<DeviceLru>();
  const uint32_t EL = h->cfg.endpoint_count, C = h->cfg.lru_capacity;
  DevLru& d = L->view;
  d.EL = EL;
  d.capacity = C;
  size_t free_b = 0, total_b = 0;
  FI_CUDA(cudaMemGetInfo(&free_b, &total_b));
  // Log: at least 4 C records (a sub-batch appends at most C; more room = rarer compaction).  Table: at least 4 C slots (C entries + C new keys of a
  // conservative sub-batch + tombstones); a table takes a batch's DISTINCT keys on top of its entries, and an
  // endpoint that attracts a popular prefix can receive a large share of a batch — so the tables get as much as
  // a quarter of the free HBM buys, up to 32 C slots (1 Mi slots = 16 MiB per endpoint at lruCapacityPerServer
  // 31 250: 17 GB for 1 024 endpoints of a B200's 180).  Option "lru_table_slots" / FI_EPP_LRU_TABLE_SLOTS pins it.
  d.L = std::max<uint32_t>(pow2_ceil32(4u * C), 64u);
  const uint32_t ts_min = d.L;
  uint32_t ts = pow2_ceil32(32u * C);
  while (ts > ts_min && (size_t)EL * (ts + 2) * sizeof(LruSlot) > free_b / 4) ts >>= 1;
  uint32_t want = h->lru_table_slots;
  if (!want)
    if (const char* ev = std::getenv("FI_EPP_LRU_TABLE_SLOTS")) want = (uint32_t)std::strtoul(ev, nullptr, 10);
  if (want) ts = std::max(ts_min, pow2_ceil32(want));
  d.TS = ts;
  d.L = std::max(d.L, d.TS / 4);
  d.insert_limit = (uint32_t)((uint64_t)d.TS * 85 / 100);
  const size_t slot_bytes = (size_t)EL * (d.TS + 2) * sizeof(LruSlot), log_bytes = (size_t)EL * d.L * sizeof(uint64_t);
  L->touch_cap = std::max<uint64_t>((uint64_t)h->cfg.max_batch * h->MP, 1u << 16);
  const size_t scratch = (size_t)L->touch_cap * (sizeof(uint32_t) + 3 * sizeof(fi_index_op));
  if (slot_bytes + log_bytes + scratch + (256u << 20) > free_b)
    return fail(h, FI_ERR_NOMEM, "device LRU does not fit in free HBM (option device_lru = 0 selects the host LRU)");
  const size_t state_words = (size_t)7 * EL + 2;
  FI_CUDA(dev_alloc(L->slots, slot_bytes));
  FI_CUDA(dev_alloc(L->log, log_bytes));
  FI_CUDA(dev_alloc(L->state, state_words * sizeof(uint32_t)));
  FI_CUDA(dev_alloc(L->ctr, 8 * sizeof(unsigned long long)));
  FI_CUDA(host_alloc(L->stat, sizeof(DeviceLru::HostStat)));
  std::memset(L->stat.get(), 0, sizeof(DeviceLru::HostStat));
  FI_CUDA(dev_alloc(L->slot_of, L->touch_cap * sizeof(uint32_t)));
  FI_CUDA(dev_alloc(L->sets, L->touch_cap * sizeof(fi_index_op)));
  FI_CUDA(dev_alloc(L->clears, 2 * L->touch_cap * sizeof(fi_index_op)));  // doomed keys + evictions
  FI_CUDA(dev_alloc(L->wcount, (size_t)h->cfg.max_batch * sizeof(uint32_t)));
  FI_CUDA(dev_alloc(L->base, (size_t)h->cfg.max_batch * sizeof(uint32_t)));
  FI_CUDA(event_create(L->ev));
  FI_CUDA(event_create(L->ev_ovf));
  FI_CUDA(cudaMemsetAsync(L->slots.get(), 0, slot_bytes, h->s_index.get()));
  FI_CUDA(cudaMemsetAsync(L->state.get(), 0, state_words * sizeof(uint32_t), h->s_index.get()));
  FI_CUDA(cudaMemsetAsync(L->ctr.get(), 0, 8 * sizeof(unsigned long long), h->s_index.get()));
  FI_CUDA(cudaEventRecord(L->ev.get(), h->s_index.get()));
  d.slots = L->slots.get();
  d.log = L->log.get();
  d.head = L->state.get();
  d.tail = d.head + EL;
  d.count = d.tail + EL;
  d.used = d.count + EL;
  d.hold = d.used + EL;
  d.dcount = d.hold + EL;
  d.ovf = d.dcount + EL;
  d.any_ovf = d.ovf + EL;
  d.error = d.any_ovf + 1;
  d.n_sets = L->ctr.get();
  d.n_maintained = L->ctr.get() + 1;
  d.n_clears = L->ctr.get() + 3;
  d.n_doomed = L->ctr.get() + 4;
  h->gen_lru++;
  *out = std::move(L);
  return FI_OK;
}

// queue the refresh of the pinned LRU status (error flag + totals) behind everything submitted so far
int lru_refresh_stat(fi_epp* h) {
  DeviceLru& L = *h->dlru;
  FI_CUDA(cudaMemcpyAsync(&L.stat->error, L.view.error, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->s_index.get()));
  FI_CUDA(cudaMemcpyAsync(&L.stat->n_sets, L.ctr.get(), 5 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->s_index.get()));
  return FI_OK;
}

// indexer.Add(chains[r], endpoints[r]) for r = 0..R-1 through the device LRU.  `chains` is a host pointer
// (copied to the device first) or, with on_device, memory the index stream can read.  The first pass is
// OPTIMISTIC: sub-batches are cut only by the scratch arrays' size, and an endpoint whose table cannot take the
// batch's distinct keys is rolled back and deferred; the deferred requests then run in a second, conservative pass
// (at most lru_capacity touches per endpoint and sub-batch: always fits).
int lru_device_add(fi_epp* h, const uint32_t* endpoints, const uint64_t* chains, bool on_device, uint32_t pitch,
                   const uint32_t* nblocks, uint32_t R, bool conservative) {
  if (!h->dlru) {
    int rc = alloc_dev_lru(h, &h->dlru);
    if (rc != FI_OK) {
      cudaGetLastError();
      return rc;
    }
  }
  DeviceLru& L = *h->dlru;
  const uint32_t EL = h->cfg.endpoint_count, lo = h->cfg.endpoint_begin;
  for (uint32_t r = 0; r < R; ++r)
    if (nblocks[r] > h->cfg.lru_capacity && endpoints[r] - lo < EL)
      return fail(h, FI_ERR_INVALID, "device LRU: a chain longer than lru_capacity");
  int rc = flush_ops(h);  // ops staged through fi_epp_index_apply come first
  if (rc != FI_OK) return rc;
  rc = check_counters(h);
  if (rc != FI_OK) return rc;
  const auto t0 = std::chrono::steady_clock::now();
  LruPlan& pl = h->lru_plan;
  // sharded pool: a sub-batch's APPEAR / VANISH transitions must fit the gossip log of one round (at most one SET per
  // touch; CLEARs: evictions <= keys added, plus doomed entries <= touches)
  const bool sharded = h->world > 1;
  const uint64_t cap_touches = sharded ? std::min<uint64_t>(L.touch_cap, kOpChunk / 2) : L.touch_cap;
  lru_plan_batch(endpoints, nblocks, R, lo, EL, conservative ? h->cfg.lru_capacity : 0xFFFFFFFFu, cap_touches, h->cfg.max_batch, &pl);
  if (pl.subs.empty() && !sharded) return FI_OK;
  const size_t K = pl.req_id.size(), nsub = pl.subs.size();
  // collective on a sharded pool: the ranks' sub-batch counts differ, every one is a gossip round for all
  uint64_t rounds = nsub;
  if (sharded) {
    rc = agree_rounds(h, nsub, &rounds);
    if (rc != FI_OK) return rc;
  }
  const GossipLog glog = gossip_log(h);
  // staging: req_id | req_ep | req_n | req_off | ep_list | ep_start[nsub][EL+1] | inc[nsub][EL]
  const size_t words = 5 * K + nsub * ((size_t)2 * EL + 1);
  FI_CUDA(cudaEventSynchronize(L.ev.get()));  // the previous call's staging (and chain copy) has been consumed
  if (words > L.plan_cap) {
    const size_t cap = words + words / 2 + 1024;
    L.plan_cap = 0;
    FI_CUDA(dev_alloc(L.d_plan, cap * sizeof(uint32_t)));
    FI_CUDA(host_alloc(L.h_plan, cap * sizeof(uint32_t)));
    L.plan_cap = cap;
  }
  uint32_t* hp = L.h_plan.get();
  if (words) {
  std::memcpy(hp, pl.req_id.data(), K * 4);
  std::memcpy(hp + K, pl.req_ep.data(), K * 4);
  std::memcpy(hp + 2 * K, pl.req_n.data(), K * 4);
  std::memcpy(hp + 3 * K, pl.req_off.data(), K * 4);
  std::memcpy(hp + 4 * K, pl.ep_list.data(), K * 4);
  std::memcpy(hp + 5 * K, pl.ep_start.data(), pl.ep_start.size() * 4);
  std::memcpy(hp + 5 * K + nsub * ((size_t)EL + 1), pl.inc.data(), pl.inc.size() * 4);
  }
  // the LRU kernels run on the index stream; like every index update they are ordered behind the picks
  // submitted so far (a pick sees the index as of its call)
  FI_CUDA(cudaStreamWaitEvent(h->s_index.get(), h->ev_pick, 0));
  if (words) FI_CUDA(cudaMemcpyAsync(L.d_plan.get(), hp, words * sizeof(uint32_t), cudaMemcpyHostToDevice, h->s_index.get()));
  h->stats.h2d_bytes += words * sizeof(uint32_t);
  const uint64_t* d_chains = chains;
  if (!on_device && K) {
    const size_t cw = (size_t)R * pitch;
    if (cw > L.chains_cap) {
      L.chains_cap = 0;
      FI_CUDA(dev_alloc(L.chains, cw * sizeof(uint64_t)));
      L.chains_cap = cw;
    }
    // only the rows the plan kept are needed; whole-range copy when most are (one DMA), row copies otherwise
    if (K * 2 >= R) {
      FI_CUDA(cudaMemcpyAsync(L.chains.get(), chains, cw * sizeof(uint64_t), cudaMemcpyHostToDevice, h->s_index.get()));
      h->stats.h2d_bytes += cw * sizeof(uint64_t);
    } else {
      for (size_t k = 0; k < K; ++k) {
        const size_t r = pl.req_id[k];
        FI_CUDA(cudaMemcpyAsync(L.chains.get() + r * pitch, chains + r * pitch, (size_t)pl.req_n[k] * sizeof(uint64_t),
                                cudaMemcpyHostToDevice, h->s_index.get()));
        h->stats.h2d_bytes += (size_t)pl.req_n[k] * sizeof(uint64_t);
      }
    }
    d_chains = L.chains.get();
  }
  const uint32_t* dp = L.d_plan.get();
  h->lru_sub_batches += nsub;
  std::vector<uint8_t> deferred;  // per request of this call: its endpoint overflowed in the optimistic pass
  std::vector<uint32_t> ovf_host;
  size_t n_deferred = 0;
  for (size_t sb = 0; sb < rounds; ++sb) {
    if (sb >= nsub) {  // (sharded) this rank is done: it only takes part in the others' gossip rounds
      rc = gossip_round(h);
      if (rc != FI_OK) return rc;
      continue;
    }
    if (sb) {  // the index counters of the previous sub-batch decide about a rebuild before more keys arrive
      rc = check_counters(h);
      if (rc != FI_OK) return rc;
    }
    const LruSubBatch& sbt = pl.subs[sb];
    LruBatch b{};
    b.req_id = dp + sbt.k_begin;
    b.req_ep = dp + K + sbt.k_begin;
    b.req_n = dp + 2 * K + sbt.k_begin;
    b.req_off = dp + 3 * K + sbt.k_begin;
    b.ep_list = dp + 4 * K + sbt.k_begin;
    b.ep_start = dp + 5 * K + sb * ((size_t)EL + 1);
    const uint32_t* inc = dp + 5 * K + nsub * ((size_t)EL + 1) + sb * (size_t)EL;
    b.chains = d_chains;
    b.pitch = pitch;
    b.K = sbt.k_end - sbt.k_begin;
    b.slot_of = L.slot_of.get();
    b.wcount = L.wcount.get();
    b.base = L.base.get();
    b.sets = L.sets.get();
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_lru_maintain(L.view, inc, false, h->s_index.get()));
    }
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_lru_touch(L.view, b, h->s_index.get()));
    }
    // did some endpoint's table refuse keys?  (one host round trip per sub-batch; everything after it is queued
    // without waiting)
    FI_CUDA(cudaMemcpyAsync(&L.stat->any_ovf, L.view.any_ovf, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->s_index.get()));
    FI_CUDA(cudaEventRecord(L.ev_ovf.get(), h->s_index.get()));
    FI_CUDA(cudaEventSynchronize(L.ev_ovf.get()));
    const bool any_ovf = L.stat->any_ovf != 0;
    if (any_ovf) {
      if (conservative) return fail(h, FI_ERR_STATE, "device LRU: overflow in a conservative sub-batch");
      {
        LaunchScope ls(h, h->s_index.get(), K_INDEX);
        FI_CUDA(launch_lru_untouch(L.view, b, h->s_index.get()));
      }
      ovf_host.resize(EL);
      FI_CUDA(cudaMemcpyAsync(ovf_host.data(), L.view.ovf, (size_t)EL * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->s_index.get()));
      FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
      if (deferred.empty()) deferred.assign(R, 0);
      for (uint32_t k = sbt.k_begin; k < sbt.k_end; ++k)
        if (ovf_host[pl.req_ep[k]]) {
          deferred[pl.req_id[k]] = 1;
          ++n_deferred;
        }
    }
    FI_CUDA(cudaMemsetAsync(L.ctr.get() + 2, 0, sizeof(unsigned long long), h->s_index.get()));
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_lru_count(L.view, b, h->s_index.get()));
    }
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_lru_scan(L.view, b, h->s_index.get()));
    }
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_lru_append(L.view, b, L.clears.get(), L.ctr.get() + 2, 2 * L.touch_cap, lo, h->s_index.get()));
    }
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_index_set(h->ix->view, h->d_ctr.get(), L.sets.get(), sbt.touches, lo, EL, h->rank, glog, h->s_index.get()));
    }
    {
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_lru_evict(L.view, L.clears.get(), L.ctr.get() + 2, 2 * L.touch_cap, lo, h->s_index.get()));
    }
    {
      // CLEARs of a sub-batch: at most one per doomed key (<= touches) and one per eviction (<= keys it added)
      const uint64_t cap = std::min<uint64_t>(2 * L.touch_cap, 2 * sbt.touches);
      LaunchScope ls(h, h->s_index.get(), K_INDEX);
      FI_CUDA(launch_index_clear_counted(h->ix->view, h->d_ctr.get(), L.clears.get(), cap, L.ctr.get() + 2, lo, EL, h->rank, glog,
                                         h->s_index.get()));
    }
    if (any_ovf) FI_CUDA(cudaMemsetAsync(L.view.ovf, 0, ((size_t)EL + 1) * sizeof(uint32_t), h->s_index.get()));  // ovf[] and any_ovf
    FI_CUDA(cudaMemcpyAsync(h->h_ctr.get(), h->d_ctr.get(), sizeof(IndexCounters), cudaMemcpyDeviceToHost, h->s_index.get()));
    FI_CUDA(cudaEventRecord(h->ev_ctr.get(), h->s_index.get()));
    h->ctr_pending = true;
    if (sharded) {  // the other ranks replay this sub-batch's transitions into their directories (and we theirs)
      rc = gossip_round(h);
      if (rc != FI_OK) return rc;
    }
  }
  rc = lru_refresh_stat(h);
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaEventRecord(h->ev_ctr.get(), h->s_index.get()));  // covers the status copy too
  FI_CUDA(cudaEventRecord(L.ev.get(), h->s_index.get()));
  h->gen_lru++;
  FI_CUDA(cudaEventRecord(h->ev_index.get(), h->s_index.get()));
  h->gen_index++;
  if (h->verbose) {
    const auto t1 = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[fi_epp] device LRU%s: %u requests (%zu kept), %zu sub-batch(es), %zu deferred, host side %.3f ms\n",
                 conservative ? " (conservative pass)" : "", R, K, nsub, n_deferred,
                 std::chrono::duration<double, std::milli>(t1 - t0).count());
  }
  h->lru_deferred += n_deferred;
  if (n_deferred || (sharded && !conservative)) {  // (sharded: every rank enters the second pass, most with nothing to do)
    std::vector<uint32_t> ep2(R);
    for (uint32_t r = 0; r < R; ++r) ep2[r] = (n_deferred && deferred[r]) ? endpoints[r] : FI_NO_ENDPOINT;
    return lru_device_add(h, ep2.data(), d_chains, true, pitch, nblocks, R, true);
  }
  return FI_OK;
}

}  // namespace fi

// The same with the chains already in device memory (e.g. the chains_out of fi_epp_pick_batch_device): nothing
// but the two small host arrays crosses PCIe.  Device LRU only.
int fi_epp_index_add_chains_device(fi_epp* h, const uint32_t* endpoints, const void* d_chains, uint32_t pitch_blocks,
                                   const uint32_t* nblocks, uint32_t R, void* stream) {
  if (!h || ((!endpoints || !nblocks) && R)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (!h->cfg.lru_capacity) return fail(h, FI_ERR_STATE, "lru_capacity is 0: no LRU");
  if (!d_chains) {  // the chains of the handle's most recent stream-ordered pick, still in its own buffer
    if (R > h->last_plain_R) return fail(h, FI_ERR_STATE, "no pick batch of that size to take the chains from");
    d_chains = h->d_chain.get();
    pitch_blocks = h->MP;
  }
  for (uint32_t r = 0; r < R; ++r) {
    if (endpoints[r] != FI_NO_ENDPOINT && endpoints[r] >= h->cfg.num_endpoints) return fail(h, FI_ERR_INVALID, "endpoint out of range");
    if (nblocks[r] > pitch_blocks) return fail(h, FI_ERR_INVALID, "nblocks[r] larger than the chain pitch");
  }
  int rc = choose_lru_mode(h);
  if (rc != FI_OK) return rc;
  if (h->lru_mode != 1) return fail(h, FI_ERR_STATE, "fi_epp_index_add_chains_device needs the device LRU");
  // the chains were produced on the caller's stream
  FI_CUDA(cudaEventRecord(h->ev_user.get(), (cudaStream_t)stream));
  FI_CUDA(cudaStreamWaitEvent(h->s_index.get(), h->ev_user.get(), 0));
  return lru_device_add(h, endpoints, static_cast<const uint64_t*>(d_chains), true, pitch_blocks, nblocks, R);
}

// Diagnostics: the device LRU's content for one endpoint, least recently used first.
int fi_epp_lru_dump(fi_epp* h, uint32_t endpoint, uint64_t* out, uint32_t cap, uint32_t* n_out) {
  if (!h || !n_out || (!out && cap)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  *n_out = 0;
  const uint32_t e = endpoint - h->cfg.endpoint_begin;
  if (e >= h->cfg.endpoint_count) return fail(h, FI_ERR_INVALID, "endpoint outside this handle's shard");
  if (h->lru_mode != 1 || !h->dlru) return h->lru_mode == 0 ? fail(h, FI_ERR_STATE, "the handle runs the host LRU") : FI_OK;
  DevPtr<uint64_t> d_out;
  DevPtr<uint32_t> d_n;
  FI_CUDA(dev_alloc(d_out, ((size_t)h->dlru->view.capacity + 1) * sizeof(uint64_t)));
  if (dev_alloc(d_n, sizeof(uint32_t)) != cudaSuccess) return fail(h, FI_ERR_NOMEM, "cudaMalloc failed");
  uint32_t n = 0;
  FI_CUDA(launch_lru_dump(h->dlru->view, e, d_out.get(), d_n.get(), h->s_index.get()));
  FI_CUDA(cudaMemcpyAsync(&n, d_n.get(), sizeof(n), cudaMemcpyDeviceToHost, h->s_index.get()));
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  if (n) FI_CUDA(cudaMemcpy(out, d_out.get(), (size_t)std::min(n, cap) * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  *n_out = n;
  return FI_OK;
}

// Diagnostics: totals of the device-resident LRU since create — out[0] SETs emitted, [1] CLEARs emitted,
// [2] doomed winners, [3] endpoint maintenance passes, [4] requests deferred to a conservative pass, [5] sub-batches.
int fi_epp_lru_counters(fi_epp* h, uint64_t out[6]) {
  if (!h || !out) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  for (int i = 0; i < 6; ++i) out[i] = 0;
  if (h->lru_mode != 1 || !h->dlru) return FI_OK;
  FI_CUDA(cudaStreamSynchronize(h->s_index.get()));
  const DeviceLru::HostStat& st = *h->dlru->stat;
  out[0] = st.n_sets;
  out[1] = st.n_clears;
  out[2] = st.n_doomed;
  out[3] = st.n_maintained;
  out[4] = h->lru_deferred;
  out[5] = h->lru_sub_batches;
  return FI_OK;
}
