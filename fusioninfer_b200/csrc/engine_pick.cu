// engine_pick.cu — picks: stream-ordered, sliced host feed, both pipelined paths, SM partition.
#include "engine.h"

namespace fi {

int upload_endpoints(fi_epp* h) {
  if (!h->eps_dirty) return FI_OK;
  FI_CUDA(cudaMemcpyAsync(h->d_eps.get(), h->eps.data(), h->eps.size() * sizeof(EndpointDev), cudaMemcpyHostToDevice, h->s_main.get()));
  h->stats.h2d_bytes += h->eps.size() * sizeof(EndpointDev);
  {
    LaunchScope ls(h, h->s_main.get(), K_OTHER);
    FI_CUDA(launch_prepare_endpoints(h->d_eps.get(), h->cfg.num_endpoints, h->cfg.endpoint_begin, h->cfg.endpoint_count, h->st,
                                     h->d_sc.get(), h->d_elig.get(), h->d_zero.get(), h->d_ztie.get(), h->s_main.get()));
  }
  // eps is pageable host memory: the copy above has been staged by the time the call returns
  h->eps_dirty = false;
  return FI_OK;
}

int upload_lora(fi_epp* h) {
  if (!h->lora_dirty) return FI_OK;
  FI_CUDA(cudaMemcpyAsync(h->d_lora.get(), h->lora.data(), h->lora.size() * sizeof(LoraDev), cudaMemcpyHostToDevice, h->s_main.get()));
  h->stats.h2d_bytes += h->lora.size() * sizeof(LoraDev);
  h->lora_dirty = false;
  return FI_OK;
}

// hash kernels for the request slice [r0, r0+R): prompts → chain (device buffers), on stream s
int run_hash(fi_epp* h, const uint8_t* d_prompts, const uint64_t* d_offsets, const uint64_t* d_h0, uint32_t r0,
             uint32_t R, cudaStream_t s) {
  uint64_t* pre = h->d_pre.get() + (size_t)r0 * h->MP;  // tiled by groups of 32 requests: r0 % 32 == 0
  uint64_t* chain = h->d_chain.get() + (size_t)r0 * h->MP;
  uint32_t* nb = h->d_nblocks.get() + r0;
  if (h->fast_hash) {
    {
      LaunchScope ls(h, s, K_HASH);
      FI_CUDA(launch_hash_blocks(d_prompts, d_offsets + r0, R, h->cfg.block_bytes, h->cfg.max_blocks, h->MP, pre, nb, 0, s));
    }
    LaunchScope ls(h, s, K_CHAIN);
    FI_CUDA(launch_chain_finalize(pre, nb, d_h0 + r0, R, h->MP, chain, false, s));
  } else {
    LaunchScope ls(h, s, K_HASH);
    FI_CUDA(launch_hash_generic(d_prompts, d_offsets + r0, d_h0 + r0, R, h->cfg.block_bytes, h->cfg.max_blocks, h->MP,
                                chain, nb, s));
  }
  return FI_OK;
}

// FI_EPP_TRACE=<call index>: print that call's kernel timeline (start/end relative to the call's start)
void dump_trace(fi_epp* h, uint32_t R) {
  if (!h->tracing) return;
  static const char* names[] = {"hash_blocks", "chain_finalize", "match_pick", "index", "other"};
  cudaStreamSynchronize(h->s_main.get());
  std::fprintf(stderr, "[fi_epp trace] rank %u call %ld: R=%u\n", h->rank, h->trace_call, R);
  for (auto& e : h->pending_ev) {
    float t0 = 0.f, t1 = 0.f;
    cudaEventSynchronize(e.b.get());
    cudaEventElapsedTime(&t0, h->ev_trace0.get(), e.a.get());
    cudaEventElapsedTime(&t1, h->ev_trace0.get(), e.b.get());
    std::fprintf(stderr, "[fi_epp trace]   r%u %-15s start %8.1f us  end %8.1f us  (%6.1f us)\n", h->rank, names[e.kind],
                 t0 * 1e3, t1 * 1e3, (t1 - t0) * 1e3);
    h->ev_pool.push_back(std::move(e.a));
    h->ev_pool.push_back(std::move(e.b));
  }
  h->pending_ev.clear();
  h->tracing = false;
}

// host prompts still to be copied (fi_epp_pick_batch): run_pick copies them, in slices when it can
struct HostFeed {
  const uint8_t* prompts;   // host
  const uint64_t* offsets;  // host, [R+1]
};

void fill_match_params(fi_epp* h, MatchParams& mp, const uint64_t* chain, const uint32_t* nb, const uint64_t* d_offsets,
                       const uint64_t* d_h0, const uint64_t* d_adapters, uint32_t R, fi_pick* out, bool local_pd) {
  mp.chain = chain;
  mp.nblocks = nb;
  mp.offsets = d_offsets;
  mp.adapters = d_adapters;
  mp.R = R;
  mp.MP = h->MP;
  mp.ix = h->ix->view;
  mp.st = h->st;
  mp.ep_begin = h->cfg.endpoint_begin;
  mp.ep_count = h->cfg.endpoint_count;
  mp.E_global = h->cfg.num_endpoints;
  mp.r_base = 0;
  mp.h0 = d_h0;
  mp.lpm = h->cfg.match_mode;
  mp.apply_pd = (h->cfg.pd_enabled && local_pd) ? 1 : 0;
  mp.pd_decode = h->cfg.pd_decode_profile;
  mp.pd_prefill = h->cfg.pd_prefill_profile;
  mp.pd_threshold = h->cfg.pd_threshold;
  mp.out = out;
  mp.probed_blocks = h->profiling ? h->d_probed.get() : nullptr;
  mp.work_counter = h->d_work.get();
  mp.zero_work_counter = 1;
  mp.lane_zero = 0;
}

// the whole pick on device buffers; result in d_out ([R][P])
int run_pick_impl(fi_epp* h, const uint8_t* d_prompts, const uint64_t* d_offsets, const uint64_t* d_h0,
                  const uint64_t* d_adapters, uint32_t R, fi_pick* d_out, const HostFeed* feed) {
  const bool sharded = h->world > 1;
  if (sharded && (h->n_sets || h->n_clears))
    return fail(h, FI_ERR_STATE, "sharded pool: index updates are collective (fi_epp_index_apply / fi_epp_index_add_chains)");
  int rc = flush_ops(h);
  if (rc != FI_OK) return rc;
  rc = check_counters(h);
  if (rc != FI_OK) return rc;
  h->tracing = !h->profiling && h->trace_call >= 0 && (long)h->stats.pick_calls == h->trace_call;
  if (h->tracing) {
    if (!h->ev_trace0) event_create(h->ev_trace0, cudaEventDefault);
    FI_CUDA(cudaStreamSynchronize(h->s_main.get()));
    FI_CUDA(cudaEventRecord(h->ev_trace0.get(), h->s_main.get()));
  }
  FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_index.get(), 0));  // every submitted op is visible
  rc = upload_endpoints(h);
  if (rc != FI_OK) return rc;
  rc = upload_lora(h);
  if (rc != FI_OK) return rc;
  if (h->pipe_seq) {  // a plain pick after pipelined submits: their stages share d_pre / d_chain with ours
    FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_a[(h->pipe_seq - 1) & 1].get(), 0));
    FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_pick, 0));  // (their matches may run on the partition's stream)
    h->part_active = false;
  }
  MatchParams mp{};
  fill_match_params(h, mp, h->d_chain.get(), h->d_nblocks.get(), d_offsets, d_h0, d_adapters, R, sharded ? h->shard->d_local.get() : d_out, !sharded);

  const uint32_t S = h->feed_slices;
  if (feed && !sharded && h->fast_hash && S > 1 && R >= 64 * S && feed->offsets[R] >= (8ull << 20)) {
    // Sliced feed.  (On DEVICE-resident inputs slicing the step is slower — DESIGN.md "What did not
    // work" — but here the copy engine is the bottleneck and the kernels of slice k hide under copy k+1.)
    uint8_t* dp = const_cast<uint8_t*>(d_prompts);
    const uint32_t per = (((R + S - 1) / S) + 31) & ~31u;
    uint32_t used = 0;
    for (uint32_t k = 0; k * per < R; ++k, ++used) {
      const uint32_t r0 = k * per, r1 = std::min(R, r0 + per);
      const uint64_t b0 = feed->offsets[r0], b1 = feed->offsets[r1];
      if (b1 > b0) FI_CUDA(cudaMemcpyAsync(dp + b0, feed->prompts + b0, b1 - b0, cudaMemcpyHostToDevice, h->s_copy.get()));
      FI_CUDA(cudaEventRecord(h->ev_copy[k].get(), h->s_copy.get()));
    }
    h->stats.h2d_bytes += feed->offsets[R];
    for (uint32_t k = 0; k < used; ++k) {
      const uint32_t r0 = k * per, Rk = std::min(per, R - r0);
      FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_copy[k].get(), 0));
      rc = run_hash(h, d_prompts, d_offsets, d_h0, r0, Rk, h->s_main.get());
      if (rc != FI_OK) return rc;
      MatchParams ms = mp;
      ms.chain = mp.chain + (size_t)r0 * h->MP;
      ms.nblocks = mp.nblocks + r0;
      ms.offsets = mp.offsets ? mp.offsets + r0 : nullptr;
      ms.adapters = mp.adapters ? mp.adapters + r0 : nullptr;
      ms.h0 = mp.h0 + r0;
      ms.r_base = r0;
      ms.R = Rk;
      ms.out = mp.out + (size_t)r0 * h->P;
      ms.work_counter = h->d_work.get() + k;
      LaunchScope ls(h, h->s_main.get(), K_MATCH);
      FI_CUDA(launch_match_pick(ms, h->sm_count, h->s_main.get()));
    }
    dump_trace(h, R);
    h->stats.pick_calls++;
    h->stats.requests += R;
    return FI_OK;
  }
  if (feed && feed->offsets[R]) {  // one copy, then the whole batch
    FI_CUDA(cudaMemcpyAsync(const_cast<uint8_t*>(d_prompts), feed->prompts, feed->offsets[R], cudaMemcpyHostToDevice, h->s_main.get()));
    h->stats.h2d_bytes += feed->offsets[R];
  }
  if (!sharded) {
    // (A sub-batch pipeline over several streams was tried and measured slower on device-resident
    // inputs — DESIGN.md "What did not work": the chain walk costs a flat serial latency at any batch
    // size and small slices pay launch/ramp overheads.)
    rc = run_hash(h, d_prompts, d_offsets, d_h0, 0, R, h->s_main.get());
    if (rc != FI_OK) return rc;
    {
      LaunchScope ls(h, h->s_main.get(), K_MATCH);
      FI_CUDA(launch_match_pick(mp, h->sm_count, h->s_main.get()));
    }
    dump_trace(h, R);
    h->stats.pick_calls++;
    h->stats.requests += R;
    return FI_OK;
  }

  // ---- endpoint-range sharded pool --------------------------------------------------------------
  Shard& sh = *h->shard;
  // Hashing: every rank needs every request's chain.  split: rank g hashes requests [g·per, (g+1)·per) and
  // the chain rows + block counts are all-gathered in place (2 KiB per request over NVLink instead of
  // re-reading 16 KiB of prompt on every rank); replicated: every rank hashes everything.
  if (h->split_hash && h->fast_hash && R >= 32 * h->world) {
    const uint32_t per = (((R + h->world - 1) / h->world) + 31) & ~31u;  // ≤ chain_rows / world
    const uint32_t r0 = std::min(R, h->rank * per), r1 = std::min(R, r0 + per);
    if (r1 > r0) {
      rc = run_hash(h, d_prompts, d_offsets, d_h0, r0, r1 - r0, h->s_main.get());
      if (rc != FI_OK) return rc;
    }
    rc = nccl_allgather(h, sh.comm.get(), h->d_chain.get() + (size_t)h->rank * per * h->MP, h->d_chain.get(),
                        (size_t)per * h->MP * sizeof(uint64_t), h->s_main.get());
    if (rc != FI_OK) return rc;
    rc = nccl_allgather(h, sh.comm.get(), h->d_nblocks.get() + (size_t)h->rank * per, h->d_nblocks.get(), (size_t)per * sizeof(uint32_t),
                        h->s_main.get());
    if (rc != FI_OK) return rc;
    h->stats.n_other += 2;  // two collectives of the step (not kernels of this library)
  } else {
    rc = run_hash(h, d_prompts, d_offsets, d_h0, 0, R, h->s_main.get());
    if (rc != FI_OK) return rc;
  }
  const bool p2p = sh.px.enabled != 0;
  if (p2p) {
    // Peer-memory exchange: match_pick stores this rank's picks as tagged words into every rank's buffer and
    // merge_picks polls per request, so the reduction has no collective call, no barrier between the ranks
    // and no host round trip.  A timeout is reported once (the kernels set the mapped host word).
    if (*sh.h_xerr) {
      *sh.h_xerr = 0;
      return fail(h, FI_ERR_COMM, "peer exchange timed out waiting for another rank");
    }
    sh.px.step += 1;
    if (sh.px.step == 0) sh.px.step = 1;  // tag 0 is the zero-initialised buffer
    mp.px = sh.px;
  }
  {
    LaunchScope ls(h, h->s_main.get(), K_MATCH);
    FI_CUDA(launch_match_pick(mp, h->sm_count, h->s_main.get()));
  }
  MergeParams mg{};
  if (p2p) {
    mg.gathered = reinterpret_cast<const fi_pick*>(sh.d_xchg.get() + sh.px.off_pick[sh.px.step & 1u]);
    mg.px = sh.px;
  } else {
    rc = nccl_allgather(h, sh.comm.get(), sh.d_local.get(), sh.d_gather.get(), (size_t)R * h->P * sizeof(fi_pick), h->s_main.get());
    if (rc != FI_OK) return rc;
    mg.gathered = sh.d_gather.get();
  }
  mg.ranks = h->world;
  mg.R = R;
  mg.P = h->P;
  mg.nblocks = h->d_nblocks.get();
  mg.offsets = d_offsets;
  mg.chain = h->d_chain.get();
  mg.h0 = d_h0;
  mg.MP = h->MP;
  mg.E_global = h->cfg.num_endpoints;
  mg.apply_pd = h->cfg.pd_enabled;
  mg.pd_decode = h->cfg.pd_decode_profile;
  mg.pd_prefill = h->cfg.pd_prefill_profile;
  mg.pd_threshold = h->cfg.pd_threshold;
  mg.out = d_out;
  {
    LaunchScope ls(h, h->s_main.get(), K_OTHER);
    FI_CUDA(launch_merge_picks(mg, h->s_main.get()));
  }
  dump_trace(h, R);
  h->stats.pick_calls++;
  h->stats.requests += R;
  return FI_OK;
}

int run_pick(fi_epp* h, const uint8_t* d_prompts, const uint64_t* d_offsets, const uint64_t* d_h0,
             const uint64_t* d_adapters, uint32_t R, fi_pick* d_out, const HostFeed* feed = nullptr) {
  int rc = run_pick_impl(h, d_prompts, d_offsets, d_h0, d_adapters, R, d_out, feed);
  if (rc != FI_OK) return rc;
  h->ev_pick = h->ev_pick_own.get();
  FI_CUDA(cudaEventRecord(h->ev_pick, h->s_main.get()));  // index updates submitted later wait for this pick
  FI_CUDA(cudaEventRecord(h->ev_plain.get(), h->s_main.get()));
  h->gen_plain++;
  h->last_plain_R = R;
  return FI_OK;
}

// ---- SM partition of the pipelined path (green contexts through the driver entry points) ------------------
struct GreenApi {
  CUresult (*DeviceGet)(CUdevice*, int) = nullptr;
  CUresult (*DeviceGetDevResource)(CUdevice, CUdevResource*, CUdevResourceType) = nullptr;
  CUresult (*DevSmResourceSplitByCount)(CUdevResource*, unsigned int*, const CUdevResource*, CUdevResource*, unsigned int,
                                        unsigned int) = nullptr;
  CUresult (*DevResourceGenerateDesc)(CUdevResourceDesc*, CUdevResource*, unsigned int) = nullptr;
  CUresult (*GreenCtxCreate)(CUgreenCtx*, CUdevResourceDesc, CUdevice, unsigned int) = nullptr;
  CUresult (*GreenCtxDestroy)(CUgreenCtx) = nullptr;
  CUresult (*GreenCtxStreamCreate)(CUstream*, CUgreenCtx, unsigned int, int) = nullptr;
  bool loaded = false, ok = false;
};
GreenApi g_green;

bool load_green_api() {
  if (g_green.loaded) return g_green.ok;
  g_green.loaded = true;
  auto get = [](const char* name, void** fn) {
    cudaDriverEntryPointQueryResult qr;
    return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &qr) == cudaSuccess && qr == cudaDriverEntryPointSuccess && *fn;
  };
  g_green.ok = get("cuDeviceGet", (void**)&g_green.DeviceGet) &&
               get("cuDeviceGetDevResource", (void**)&g_green.DeviceGetDevResource) &&
               get("cuDevSmResourceSplitByCount", (void**)&g_green.DevSmResourceSplitByCount) &&
               get("cuDevResourceGenerateDesc", (void**)&g_green.DevResourceGenerateDesc) &&
               get("cuGreenCtxCreate", (void**)&g_green.GreenCtxCreate) &&
               get("cuGreenCtxDestroy", (void**)&g_green.GreenCtxDestroy) &&
               get("cuGreenCtxStreamCreate", (void**)&g_green.GreenCtxStreamCreate);
  cudaGetLastError();
  return g_green.ok;
}

void green_ctx_destroy(CUgreenCtx c) { g_green.GreenCtxDestroy(c); }

// Try to split the GPU (once per setting of part_want); on any failure the pipelined path keeps running
// unpartitioned.
void setup_partition(fi_epp* h) {
  if (h->part_tried) return;
  h->part_tried = true;
  if (h->part_want <= 0 || h->world > 1 || !load_green_api()) return;
  CUdevice dev;
  CUdevResource all{}, grp{}, rem{};
  unsigned int nb = 1;
  if (g_green.DeviceGet(&dev, h->cfg.device) != CUDA_SUCCESS) return;
  if (g_green.DeviceGetDevResource(dev, &all, CU_DEV_RESOURCE_TYPE_SM) != CUDA_SUCCESS) return;
  if (g_green.DevSmResourceSplitByCount(&grp, &nb, &all, &rem, 0, (unsigned)h->part_want) != CUDA_SUCCESS || nb != 1) return;
  if (grp.sm.smCount < 8 || rem.sm.smCount < 64) return;
  CUdevResourceDesc dw = nullptr, dm = nullptr;
  if (g_green.DevResourceGenerateDesc(&dw, &grp, 1) != CUDA_SUCCESS) return;
  if (g_green.DevResourceGenerateDesc(&dm, &rem, 1) != CUDA_SUCCESS) return;
  auto pt = std::make_unique<Partition>();
  CUgreenCtx gw = nullptr, gm = nullptr;
  if (g_green.GreenCtxCreate(&gw, dw, dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) return;
  pt->gctx_walk.reset(gw);
  if (g_green.GreenCtxCreate(&gm, dm, dev, CU_GREEN_CTX_DEFAULT_STREAM) != CUDA_SUCCESS) return;
  pt->gctx_main.reset(gm);
  // hash_blocks(k+2) and match_pick(k) become runnable at the same moment (both wait for match_pick(k-1)) and share
  // the big partition; which of them gets its CTAs resident first decided the step — 116 us on some boxes, 138 us
  // on others with the same code.  Stream priorities make the block scheduler prefer one of them whenever SMs free
  // up (FI_EPP_PIPE_PRIO=match | hash | none).
  int prio_lo = 0, prio_hi = 0;
  cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);  // lo = least (numerically greatest), hi = greatest priority
  int pa = 0, pb = 0;
  const char* pe = std::getenv("FI_EPP_PIPE_PRIO");
  const std::string prio = pe ? pe : "none";  // (measured on a 116-us box: none 116.1, hash 116.2, match 121.2 us)
  if (prio == "match") {
    pa = prio_lo;
    pb = prio_hi;
  } else if (prio == "hash") {
    pa = prio_hi;
    pb = prio_lo;
  }
  CUstream sw = nullptr, sa = nullptr, sb = nullptr;
  if (g_green.GreenCtxStreamCreate(&sw, gw, CU_STREAM_NON_BLOCKING, 0) != CUDA_SUCCESS) return;
  pt->s_pw.reset(sw);
  if (g_green.GreenCtxStreamCreate(&sa, gm, CU_STREAM_NON_BLOCKING, pa) != CUDA_SUCCESS) return;
  pt->s_pa.reset(sa);
  if (g_green.GreenCtxStreamCreate(&sb, gm, CU_STREAM_NON_BLOCKING, pb) != CUDA_SUCCESS) return;
  pt->s_pb.reset(sb);
  bool ok = dev_alloc(pt->d_pre2, (size_t)h->chain_rows * h->MP * sizeof(uint64_t)) == cudaSuccess &&
            dev_alloc(pt->d_nblocks3, (size_t)h->cfg.max_batch * sizeof(uint32_t)) == cudaSuccess;
  for (Event* e : {&pt->ev_h[0], &pt->ev_h[1], &pt->ev_b3[0], &pt->ev_b3[1], &pt->ev_b3[2], &pt->ev_up})
    ok = ok && event_create(*e) == cudaSuccess;
  if (!ok) {
    cudaGetLastError();
    return;
  }
  pt->walk_sms = (int)grp.sm.smCount;
  pt->main_sms = (int)rem.sm.smCount;
  h->part = std::move(pt);
  if (h->verbose)
    std::fprintf(stderr, "[fi_epp] pipelined path: SM partition %d (chain walk) + %d (hashing, matching), three batches in flight\n",
                 h->part->walk_sms, h->part->main_sms);
}

// Pipelined device path on the partitioned GPU: hash(k) and match(k) on the big partition's two streams,
// chain(k) on the walker partition.  Buffers: pre[2] and chain[2] by batch parity, nblocks[3] by k mod 3 (hash(k+2)
// writes its block counts while match(k) still reads its own).
// the second buffer slot of the pipelined path, built at the first submit
int alloc_pipe_slot(fi_epp* h, std::unique_ptr<PipeSlot>* out) {
  auto ps = std::make_unique<PipeSlot>();
  FI_CUDA(dev_alloc(ps->chain, (size_t)h->cfg.max_batch * h->MP * sizeof(uint64_t)));
  FI_CUDA(dev_alloc(ps->nblocks, (size_t)h->cfg.max_batch * sizeof(uint32_t)));
  *out = std::move(ps);
  return FI_OK;
}

int submit_pick_partitioned(fi_epp* h, const uint8_t* d_prompts, const uint64_t* d_offsets, const uint64_t* d_h0, uint32_t R,
                            fi_pick* d_out, cudaStream_t us) {
  Partition& pt = *h->part;
  const uint64_t k = h->pipe_seq;
  const uint32_t s2 = (uint32_t)(k & 1), s3 = (uint32_t)(k % 3);
  uint64_t* pre = s2 ? pt.d_pre2.get() : h->d_pre.get();
  uint64_t* chain = s2 ? h->slot2->chain.get() : h->d_chain.get();
  uint32_t* nb = s3 == 0 ? h->d_nblocks.get() : (s3 == 1 ? h->slot2->nblocks.get() : pt.d_nblocks3.get());
  // ---- hash(k): inputs ready in the caller's stream order; pre[s2] free once chain(k-2) has read it, nb[s3] once
  // match(k-3) has; d_pre / d_chain are shared with stream-ordered picks and with the device LRU's reads
  FI_CUDA(cudaEventRecord(h->ev_in.get(), us));
  FI_CUDA(cudaStreamWaitEvent(pt.s_pa.get(), h->ev_in.get(), 0));
  if (h->seen_plain != h->gen_plain) {
    FI_CUDA(cudaStreamWaitEvent(pt.s_pa.get(), h->ev_plain.get(), 0));
    h->seen_plain = h->gen_plain;
  }
  if (h->dlru && h->seen_lru != h->gen_lru) {
    FI_CUDA(cudaStreamWaitEvent(pt.s_pa.get(), h->dlru->ev.get(), 0));
    h->seen_lru = h->gen_lru;
  }
  if (h->part_seq >= 2) FI_CUDA(cudaStreamWaitEvent(pt.s_pa.get(), h->ev_a[s2].get(), 0));
  if (h->part_seq >= 3) FI_CUDA(cudaStreamWaitEvent(pt.s_pa.get(), pt.ev_b3[s3].get(), 0));
  {
    LaunchScope ls(h, pt.s_pa.get(), K_HASH);
    // (the kernel also zeroes the request-queue counter of this batch's match_pick: one runtime call less per batch)
    // hash_blocks runs as 4 persistent CTAs per SM here (FI_EPP_PIPE_HASH_CTAS / option "pipe_hash_ctas" overrides;
    // a large value = one CTA per request).  With one CTA per request the step is bimodal: 116 us on most boxes,
    // 138 us on others (among them the 8-GPU node) with the same binary — depending on which of the two kernels
    // gets its CTAs resident first, hash_blocks' 16 384 short CTAs and match_pick's 324 long ones (80 registers
    // x 256 threads x 3 per SM) lock each other out of the SMs.  Four hashing CTAs (32 K registers) always leave
    // room for one matching CTA next to them: 122.6-123.3 us on both kinds of box.
    const uint32_t hash_ctas = h->pipe_hash_ctas ? h->pipe_hash_ctas : 4u;
    FI_CUDA(launch_hash_blocks(d_prompts, d_offsets, R, h->cfg.block_bytes, h->cfg.max_blocks, h->MP, pre, nb,
                               hash_ctas * (uint32_t)pt.main_sms, pt.s_pa.get(), h->d_work.get() + 8 + s3));
  }
  FI_CUDA(cudaEventRecord(pt.ev_h[s2].get(), pt.s_pa.get()));
  // ---- chain(k) on its own SMs: chain[s2] free once match(k-2) has read it
  FI_CUDA(cudaStreamWaitEvent(pt.s_pw.get(), pt.ev_h[s2].get(), 0));
  if (h->part_seq >= 2) FI_CUDA(cudaStreamWaitEvent(pt.s_pw.get(), pt.ev_b3[(k + 1) % 3].get(), 0));  // (k - 2) mod 3
  {
    LaunchScope ls(h, pt.s_pw.get(), K_CHAIN);
    const bool compact = h->part_compact < 0 ? pt.walk_sms < 24 : h->part_compact != 0;
    FI_CUDA(launch_chain_finalize(pre, nb, d_h0, R, h->MP, chain, compact, pt.s_pw.get()));
  }
  FI_CUDA(cudaEventRecord(h->ev_a[s2].get(), pt.s_pw.get()));
  // ---- match(k): every submitted index op and pod-state update is visible
  if (h->eps_dirty || h->lora_dirty) {
    int rc = upload_endpoints(h);  // (on s_main)
    if (rc != FI_OK) return rc;
    rc = upload_lora(h);
    if (rc != FI_OK) return rc;
    FI_CUDA(cudaEventRecord(pt.ev_up.get(), h->s_main.get()));
    FI_CUDA(cudaStreamWaitEvent(pt.s_pb.get(), pt.ev_up.get(), 0));
  }
  if (h->seen_index != h->gen_index) {
    FI_CUDA(cudaStreamWaitEvent(pt.s_pb.get(), h->ev_index.get(), 0));
    h->seen_index = h->gen_index;
  }
  FI_CUDA(cudaStreamWaitEvent(pt.s_pb.get(), h->ev_a[s2].get(), 0));
  MatchParams mp{};
  fill_match_params(h, mp, chain, nb, d_offsets, d_h0, nullptr, R, d_out, true);
  mp.work_counter = h->d_work.get() + 8 + s3;
  mp.max_ctas_per_sm = h->pipe_match_ctas;
  mp.zero_work_counter = 0;  // hash_blocks of this batch did
  {
    LaunchScope ls(h, pt.s_pb.get(), K_MATCH);
    FI_CUDA(launch_match_pick(mp, pt.main_sms, pt.s_pb.get()));
  }
  FI_CUDA(cudaEventRecord(pt.ev_b3[s3].get(), pt.s_pb.get()));
  h->ev_pick = pt.ev_b3[s3].get();
  h->pipe_seq++;
  h->part_seq++;
  h->stats.pick_calls++;
  h->stats.requests += R;
  return FI_OK;
}

// Pipelined device path: enqueue one batch.  Stage A on s_a, stage B on s_main (see fi_epp::s_a).
int submit_pick(fi_epp* h, const uint8_t* d_prompts, const uint64_t* d_offsets, const uint64_t* d_h0, uint32_t R,
                fi_pick* d_out, cudaStream_t us) {
  int rc = flush_ops(h);
  if (rc != FI_OK) return rc;
  rc = check_counters(h);
  if (rc != FI_OK) return rc;
  if (!h->slot2) {
    rc = alloc_pipe_slot(h, &h->slot2);
    if (rc != FI_OK) return rc;
  }
  setup_partition(h);
  if (h->part && h->trace_call < 0) {
    if (!h->part_active) {
      // switching from the two-stream pipeline (or first use): everything in flight there is ordered before us
      // through ev_plain / ev_pick; the slot events of the partitioned pipeline start fresh
      FI_CUDA(cudaStreamWaitEvent(h->part->s_pa.get(), h->ev_pick, 0));
      FI_CUDA(cudaStreamWaitEvent(h->part->s_pw.get(), h->ev_pick, 0));
      h->part_active = true;
      h->part_seq = 0;
      h->seen_index = h->seen_plain = h->seen_lru = ~0ull;
    }
    return submit_pick_partitioned(h, d_prompts, d_offsets, d_h0, R, d_out, us);
  }
  // FI_EPP_TRACE=<call>: timeline of three consecutive pipelined batches (printed by fi_epp_pick_wait)
  if (!h->profiling && h->trace_call >= 0 && (long)h->stats.pick_calls >= h->trace_call &&
      (long)h->stats.pick_calls < h->trace_call + 3) {
    if ((long)h->stats.pick_calls == h->trace_call) {
      if (!h->ev_trace0) event_create(h->ev_trace0, cudaEventDefault);
      FI_CUDA(cudaStreamSynchronize(h->s_main.get()));
      FI_CUDA(cudaStreamSynchronize(h->s_a.get()));
      FI_CUDA(cudaEventRecord(h->ev_trace0.get(), h->s_main.get()));
      FI_CUDA(cudaStreamWaitEvent(h->s_a.get(), h->ev_trace0.get(), 0));
    }
    h->tracing = true;
  } else if (h->tracing && (long)h->stats.pick_calls >= h->trace_call + 3) {
    h->tracing = false;  // events stay queued until the dump
  }
  const uint32_t slot = (uint32_t)(h->pipe_seq & 1);
  uint64_t* chain = slot ? h->slot2->chain.get() : h->d_chain.get();
  uint32_t* nb = slot ? h->slot2->nblocks.get() : h->d_nblocks.get();
  // ---- stage A: inputs are ready in the caller's stream order; the slot's buffers are free once the
  // match of two batches ago is done; d_pre is free once the previous plain pick (if any) is done
  FI_CUDA(cudaEventRecord(h->ev_in.get(), us));
  FI_CUDA(cudaStreamWaitEvent(h->s_a.get(), h->ev_in.get(), 0));
  if (h->pipe_seq >= 2) FI_CUDA(cudaStreamWaitEvent(h->s_a.get(), h->ev_b[slot].get(), 0));
  FI_CUDA(cudaStreamWaitEvent(h->s_a.get(), h->ev_plain.get(), 0));
  if (h->dlru) FI_CUDA(cudaStreamWaitEvent(h->s_a.get(), h->dlru->ev.get(), 0));  // a device-LRU Add may still be reading d_chain
  {
    LaunchScope ls(h, h->s_a.get(), K_HASH);
    // The SM split of the pipeline: this batch's block hashing runs BESIDE the previous batch's match_pick —
    // hash_blocks as at most pipe_hash_ctas CTAs per SM, match_pick as at most pipe_match_ctas (its three CTAs of
    // 79 registers would leave no room) — instead of one after the other.
    FI_CUDA(launch_hash_blocks(d_prompts, d_offsets, R, h->cfg.block_bytes, h->cfg.max_blocks, h->MP, h->d_pre.get(), nb,
                               h->pipe_hash_ctas * (uint32_t)h->sm_count, h->s_a.get()));
  }
  // The chain walk is serial latency — a warp per scheduler that wants an issue slot every few cycles — and
  // runs 3x slower next to a busy kernel (measured: 30 -> 100 us under match_pick), so it waits for the
  // previous batch's match to drain; what overlaps is this batch's block hashing with that match.
  if (h->pipe_seq >= 1) FI_CUDA(cudaStreamWaitEvent(h->s_a.get(), h->ev_b[slot ^ 1u].get(), 0));
  {
    LaunchScope ls(h, h->s_a.get(), K_CHAIN);
    FI_CUDA(launch_chain_finalize(h->d_pre.get(), nb, d_h0, R, h->MP, chain, false, h->s_a.get()));
  }
  FI_CUDA(cudaEventRecord(h->ev_a[slot].get(), h->s_a.get()));
  // ---- stage B
  FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_index.get(), 0));  // every submitted op is visible
  rc = upload_endpoints(h);
  if (rc != FI_OK) return rc;
  rc = upload_lora(h);
  if (rc != FI_OK) return rc;
  FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_a[slot].get(), 0));
  MatchParams mp{};
  fill_match_params(h, mp, chain, nb, d_offsets, d_h0, nullptr, R, d_out, true);
  mp.work_counter = h->d_work.get() + 8 + slot;
  mp.max_ctas_per_sm = h->pipe_match_ctas;
  {
    LaunchScope ls(h, h->s_main.get(), K_MATCH);
    FI_CUDA(launch_match_pick(mp, h->sm_count, h->s_main.get()));
  }
  FI_CUDA(cudaEventRecord(h->ev_b[slot].get(), h->s_main.get()));
  h->ev_pick = h->ev_pick_own.get();
  FI_CUDA(cudaEventRecord(h->ev_pick, h->s_main.get()));
  h->pipe_seq++;
  h->stats.pick_calls++;
  h->stats.requests += R;
  return FI_OK;
}

}  // namespace fi

static int check_batch(fi_epp* h, const uint64_t* offsets, uint32_t R, uint64_t* total) {
  if (R > h->cfg.max_batch) return fail(h, FI_ERR_CAPACITY, "batch larger than max_batch");
  if (offsets[0] != 0) return fail(h, FI_ERR_INVALID, "offsets[0] must be 0");
  for (uint32_t r = 0; r < R; ++r)
    if (offsets[r + 1] < offsets[r]) return fail(h, FI_ERR_INVALID, "offsets must be non-decreasing");
  *total = offsets[R];
  if (*total > h->cfg.max_prompt_bytes) return fail(h, FI_ERR_CAPACITY, "prompt bytes larger than max_prompt_bytes");
  return FI_OK;
}

static int stage_inputs(fi_epp* h, const uint8_t* prompts, const uint64_t* offsets, const uint64_t* h0, uint32_t R,
                        uint64_t total, bool copy_prompts = true) {
  std::memcpy(h->h_offsets.get(), offsets, (size_t)(R + 1) * sizeof(uint64_t));
  std::memcpy(h->h_h0.get(), h0, (size_t)R * sizeof(uint64_t));
  FI_CUDA(cudaMemcpyAsync(h->d_offsets.get(), h->h_offsets.get(), (size_t)(R + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, h->s_main.get()));
  FI_CUDA(cudaMemcpyAsync(h->d_h0.get(), h->h_h0.get(), (size_t)R * sizeof(uint64_t), cudaMemcpyHostToDevice, h->s_main.get()));
  if (total && copy_prompts) {
    FI_CUDA(cudaMemcpyAsync(h->d_prompts.get(), prompts, total, cudaMemcpyHostToDevice, h->s_main.get()));
    h->stats.h2d_bytes += total;
  }
  h->stats.h2d_bytes += (size_t)(2 * R + 1) * sizeof(uint64_t);
  return FI_OK;
}

static int copy_chains_out(fi_epp* h, uint64_t* chains_out, uint32_t R, cudaMemcpyKind kind, cudaStream_t s) {
  const size_t row = (size_t)h->cfg.max_blocks * sizeof(uint64_t);
  FI_CUDA(cudaMemcpy2DAsync(chains_out, row, h->d_chain.get(), (size_t)h->MP * sizeof(uint64_t), row, R, kind, s));
  if (kind == cudaMemcpyDeviceToHost) h->stats.d2h_bytes += row * R;
  return FI_OK;
}

int fi_epp_hash_batch(fi_epp* h, const uint8_t* prompts, const uint64_t* offsets, const uint64_t* h0, uint32_t R,
                      uint64_t* chains_out, uint32_t* nblocks_out) {
  if (!h || !offsets || (!h0 && R) || (!prompts && R && offsets[R])) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (R == 0) return FI_OK;
  uint64_t total = 0;
  int rc = check_batch(h, offsets, R, &total);
  if (rc != FI_OK) return rc;
  rc = stage_inputs(h, prompts, offsets, h0, R, total);
  if (rc != FI_OK) return rc;
  if (h->pipe_seq)  // a pipelined batch's stage A (on s_a) shares d_pre with us
    FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_a[(h->pipe_seq - 1) & 1].get(), 0));
  if (h->dlru) FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->dlru->ev.get(), 0));  // a device-LRU Add may still be reading d_chain
  h->last_plain_R = 0;  // d_chain no longer holds a pick batch's chains
  rc = run_hash(h, h->d_prompts.get(), h->d_offsets.get(), h->d_h0.get(), 0, R, h->s_main.get());
  if (rc != FI_OK) return rc;
  if (chains_out) {
    rc = copy_chains_out(h, chains_out, R, cudaMemcpyDeviceToHost, h->s_main.get());
    if (rc != FI_OK) return rc;
  }
  if (nblocks_out) {
    FI_CUDA(cudaMemcpyAsync(h->h_nblocks.get(), h->d_nblocks.get(), (size_t)R * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->s_main.get()));
    h->stats.d2h_bytes += (size_t)R * sizeof(uint32_t);
  }
  FI_CUDA(cudaStreamSynchronize(h->s_main.get()));
  if (nblocks_out) std::memcpy(nblocks_out, h->h_nblocks.get(), (size_t)R * sizeof(uint32_t));
  return FI_OK;
}

int fi_epp_pick_batch(fi_epp* h, const uint8_t* prompts, const uint64_t* offsets, const uint64_t* h0, uint32_t R,
                      fi_pick* out, uint64_t* chains_out) {
  return fi_epp_pick_batch_lora(h, prompts, offsets, h0, nullptr, R, out, chains_out);
}

int fi_epp_pick_batch_lora(fi_epp* h, const uint8_t* prompts, const uint64_t* offsets, const uint64_t* h0,
                           const uint64_t* adapters, uint32_t R, fi_pick* out, uint64_t* chains_out) {
  if (!h || !offsets || (!h0 && R) || (!out && R) || (!prompts && R && offsets[R])) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (R == 0) return FI_OK;
  uint64_t total = 0;
  int rc = check_batch(h, offsets, R, &total);
  if (rc != FI_OK) return rc;
  rc = stage_inputs(h, prompts, offsets, h0, R, total, /*copy_prompts=*/false);  // run_pick feeds the prompts
  if (rc != FI_OK) return rc;
  if (adapters) {
    std::memcpy(h->h_adapters.get(), adapters, (size_t)R * sizeof(uint64_t));
    FI_CUDA(cudaMemcpyAsync(h->d_adapters.get(), h->h_adapters.get(), (size_t)R * sizeof(uint64_t), cudaMemcpyHostToDevice, h->s_main.get()));
    h->stats.h2d_bytes += (size_t)R * sizeof(uint64_t);
  }
  const HostFeed feed{prompts, offsets};
  rc = run_pick(h, h->d_prompts.get(), h->d_offsets.get(), h->d_h0.get(), adapters ? h->d_adapters.get() : nullptr, R, h->d_picks.get(), &feed);
  if (rc != FI_OK) return rc;
  const size_t pb = (size_t)R * h->P * sizeof(fi_pick);
  FI_CUDA(cudaMemcpyAsync(h->h_picks.get(), h->d_picks.get(), pb, cudaMemcpyDeviceToHost, h->s_main.get()));
  h->stats.d2h_bytes += pb;
  if (chains_out) {
    rc = copy_chains_out(h, chains_out, R, cudaMemcpyDeviceToHost, h->s_main.get());
    if (rc != FI_OK) return rc;
  }
  FI_CUDA(cudaStreamSynchronize(h->s_main.get()));
  if (h->shard && h->shard->h_xerr && *h->shard->h_xerr) {  // reported once; the tags are monotonic, so later steps can succeed again
    *h->shard->h_xerr = 0;
    return fail(h, FI_ERR_COMM, "peer exchange timed out waiting for another rank");
  }
  std::memcpy(out, h->h_picks.get(), pb);
  return FI_OK;
}

int fi_epp_pick_batch_device(fi_epp* h, const void* d_prompts, const void* d_offsets, const void* d_h0, uint32_t R,
                             uint64_t total_prompt_bytes, void* d_out, void* d_chains_out, void* stream) {
  return fi_epp_pick_batch_device_lora(h, d_prompts, d_offsets, d_h0, nullptr, R, total_prompt_bytes, d_out, d_chains_out,
                                       stream);
}

int fi_epp_pick_batch_device_lora(fi_epp* h, const void* d_prompts, const void* d_offsets, const void* d_h0,
                                  const void* d_adapters, uint32_t R, uint64_t total_prompt_bytes, void* d_out,
                                  void* d_chains_out, void* stream) {
  if (!h || !d_offsets || (!d_h0 && R) || (!d_out && R)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (R == 0) return FI_OK;
  if (R > h->cfg.max_batch) return fail(h, FI_ERR_CAPACITY, "batch larger than max_batch");
  (void)total_prompt_bytes;  // inputs stay where they are: no staging copy, no capacity limit
  cudaStream_t us = (cudaStream_t)stream;
  FI_CUDA(cudaEventRecord(h->ev_user.get(), us));
  FI_CUDA(cudaStreamWaitEvent(h->s_main.get(), h->ev_user.get(), 0));
  int rc = run_pick(h, (const uint8_t*)d_prompts, (const uint64_t*)d_offsets, (const uint64_t*)d_h0,
                    (const uint64_t*)d_adapters, R, (fi_pick*)d_out);
  if (rc != FI_OK) return rc;
  if (d_chains_out) {
    rc = copy_chains_out(h, (uint64_t*)d_chains_out, R, cudaMemcpyDeviceToDevice, h->s_main.get());
    if (rc != FI_OK) return rc;
  }
  FI_CUDA(cudaEventRecord(h->ev_done.get(), h->s_main.get()));
  FI_CUDA(cudaStreamWaitEvent(us, h->ev_done.get(), 0));
  return FI_OK;
}

int fi_epp_pick_submit(fi_epp* h, const void* d_prompts, const void* d_offsets, const void* d_h0, uint32_t R,
                       uint64_t total_prompt_bytes, void* d_out, void* stream) {
  if (!h || !d_offsets || (!d_h0 && R) || (!d_out && R)) return FI_ERR_INVALID;
  bool plain;
  {
    std::lock_guard<std::mutex> lk(h->mu);
    plain = h->world > 1 || !h->fast_hash;  // sharded pools and odd block sizes: the stream-ordered path
  }
  if (plain) return fi_epp_pick_batch_device(h, d_prompts, d_offsets, d_h0, R, total_prompt_bytes, d_out, nullptr, stream);
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  if (R == 0) return FI_OK;
  if (R > h->cfg.max_batch) return fail(h, FI_ERR_CAPACITY, "batch larger than max_batch");
  return submit_pick(h, (const uint8_t*)d_prompts, (const uint64_t*)d_offsets, (const uint64_t*)d_h0, R, (fi_pick*)d_out,
                     (cudaStream_t)stream);
}

// out[0] = 1 if the pipelined path (fi_epp_pick_submit) runs on a partitioned GPU, out[1] / out[2] = SMs of the chain-walk
// partition / of the hashing + matching partition (0 when unpartitioned or not yet used).
int fi_epp_pipeline_info(fi_epp* h, int32_t out[3]) {
  if (!h || !out) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  out[0] = h->part ? 1 : 0;
  out[1] = h->part ? h->part->walk_sms : 0;
  out[2] = h->part ? h->part->main_sms : 0;
  return FI_OK;
}

int fi_epp_pick_wait(fi_epp* h, void* stream) {
  if (!h) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  FI_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, h->ev_pick, 0));  // s_main runs the batches in order
  if (!h->profiling && !h->pending_ev.empty() && h->ev_trace0) {
    h->tracing = true;
    dump_trace(h, 0);
  }
  return FI_OK;
}
