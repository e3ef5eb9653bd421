// engine.cu — host side of libfi_epp (handle and parts: engine.h): create, destroy, options, stats, other entry points.
#include "engine.h"

namespace fi {

void drain_profile(fi_epp* h) {
  for (auto& e : h->pending_ev) {
    float ms = 0.f;
    if (cudaEventSynchronize(e.b.get()) == cudaSuccess && cudaEventElapsedTime(&ms, e.a.get(), e.b.get()) == cudaSuccess) {
      switch (e.kind) {
        case K_HASH: h->stats.ms_hash_blocks += ms; h->stats.n_hash_blocks++; break;
        case K_CHAIN: h->stats.ms_chain_probe += ms; h->stats.n_chain_probe++; break;
        case K_MATCH: h->stats.ms_match_pick += ms; h->stats.n_match_pick++; break;
        case K_INDEX: h->stats.ms_index_apply += ms; h->stats.n_index_apply++; break;
        default: h->stats.ms_other += ms; h->stats.n_other++; break;
      }
    }
    h->ev_pool.push_back(std::move(e.a));
    h->ev_pool.push_back(std::move(e.b));
  }
  h->pending_ev.clear();
}

int validate_config(const fi_epp_config& c, std::string* err) {
  auto bad = [&](const char* m) {
    *err = m;
    return FI_ERR_INVALID;
  };
  if (c.struct_size != sizeof(fi_epp_config)) return bad("struct_size mismatch");
  if (c.abi_version != FI_EPP_ABI_VERSION) return bad("abi_version mismatch");
  if (c.block_bytes == 0 || c.block_bytes > (1u << 20)) return bad("block_bytes out of range");
  if (c.max_blocks == 0 || c.max_blocks > FI_EPP_MAX_BLOCKS) return bad("max_blocks out of range");
  if (c.num_endpoints == 0) return bad("num_endpoints == 0");
  if (c.endpoint_count == 0 || (uint64_t)c.endpoint_begin + c.endpoint_count > c.num_endpoints)
    return bad("endpoint shard out of range");
  if (c.endpoint_count > 4096) return bad("more than 4096 local endpoints: shard the pool by endpoint range");
  if (c.match_mode != FI_MATCH_UPSTREAM && c.match_mode != FI_MATCH_LPM) return bad("bad match_mode");
  if (c.max_batch == 0) return bad("max_batch == 0");
  if (c.n_profiles == 0 || c.n_profiles > FI_EPP_MAX_PROFILES) return bad("n_profiles out of range");
  for (uint32_t p = 0; p < c.n_profiles; ++p) {
    if (c.profiles[p].n_scorers > FI_EPP_MAX_SCORERS) return bad("n_scorers out of range");
    if (c.profiles[p].n_more_filters > FI_EPP_MAX_FILTERS - 1) return bad("n_more_filters out of range");
    for (uint32_t f = 0; f < c.profiles[p].n_more_filters; ++f)
      if (c.profiles[p].more_filters[f] == 0) return bad("a by-label filter without label bits admits nothing");
    for (uint32_t s = 0; s < c.profiles[p].n_scorers; ++s) {
      const uint32_t k = c.profiles[p].scorers[s].kind;
      if (k != FI_SCORER_PREFIX && k != FI_SCORER_KV_UTIL && k != FI_SCORER_QUEUE && k != FI_SCORER_LORA)
        return bad("unknown scorer kind");
      if (c.profiles[p].scorers[s].weight < 0) return bad("scorer weights must be >= 0");
    }
  }
  if (c.pd_enabled) {
    if (c.pd_decode_profile >= c.n_profiles || c.pd_prefill_profile >= c.n_profiles) return bad("pd profile index out of range");
    if (!(c.pd_threshold == c.pd_threshold)) return bad("pd_threshold is NaN");
  }
  if (c.index_slots) {
    if (c.index_slots < 64 || (c.index_slots & (c.index_slots - 1))) return bad("index_slots must be a power of two >= 64");
    if (c.index_slots > 0xFFFFFF00ull) return bad("index_slots too large");
  }
  return FI_OK;
}

}  // namespace fi

// =============================================================================
// C ABI
// =============================================================================
extern "C" {

uint32_t fi_epp_abi_version(void) { return FI_EPP_ABI_VERSION; }

const char* fi_epp_status_string(int s) {
  switch (s) {
    case FI_OK: return "ok";
    case FI_ERR_INVALID: return "invalid argument";
    case FI_ERR_CUDA: return "CUDA error (no CPU fallback exists)";
    case FI_ERR_NOMEM: return "out of memory";
    case FI_ERR_CAPACITY: return "capacity exceeded";
    case FI_ERR_STATE: return "invalid state";
    case FI_ERR_COMM: return "communicator error";
    case FI_ERR_CONFIG: return "EndpointPickerConfig rejected";
    default: return "unknown status";
  }
}

int fi_epp_config_default(fi_epp_config* c) {
  if (!c) return FI_ERR_INVALID;
  std::memset(c, 0, sizeof(*c));
  c->struct_size = sizeof(*c);
  c->abi_version = FI_EPP_ABI_VERSION;
  c->device = 0;
  c->block_bytes = 64;     // 16 uint32 tokens (SURVEY.md §8d); the reference YAML overrides it (strategy.go:57)
  c->max_blocks = 256;     // strategy.go:58
  c->lru_capacity = 31250; // strategy.go:59
  c->num_endpoints = 1;
  c->endpoint_begin = 0;
  c->endpoint_count = 1;
  c->match_mode = FI_MATCH_UPSTREAM;
  c->max_batch = 1024;
  c->max_prompt_bytes = 0;  // 0 = max_batch * block_bytes * max_blocks
  c->index_slots = 0;
  c->n_profiles = 1;  // generatePrefixCacheConfig: profile "default" = picker + prefix scorer weight 100
  std::snprintf(c->profiles[0].name, sizeof(c->profiles[0].name), "default");
  c->profiles[0].n_scorers = 1;
  c->profiles[0].scorers[0].kind = FI_SCORER_PREFIX;
  c->profiles[0].scorers[0].weight = 100;  // strategy.go:66
  return FI_OK;
}

int fi_epp_model_seed(const void* model, size_t model_len, const void* salt, size_t salt_len, uint64_t* h0) {
  if (!h0 || (!model && model_len) || (!salt && salt_len)) return FI_ERR_INVALID;
  if (model_len + salt_len > 0x7FFFFFFFull) return FI_ERR_INVALID;
  std::vector<uint8_t> buf(model_len + salt_len);
  if (model_len) std::memcpy(buf.data(), model, model_len);
  if (salt_len) std::memcpy(buf.data() + model_len, salt, salt_len);
  *h0 = xxh64_bytes(buf.data(), (uint32_t)buf.size());
  return FI_OK;
}

void* fi_epp_pinned_alloc(size_t bytes) {
  HostPtr<void> p;
  if (host_alloc(p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  return p.release();
}
void fi_epp_pinned_free(void* p) { HostPtr<void> released_here(p); }

const char* fi_epp_last_error(const fi_epp* h) { return h ? h->err.c_str() : "null handle"; }

// Every resource of the handle has an owner that releases it; the order of the members of fi_epp is the order
// of release.
void fi_epp_destroy(fi_epp* h) {
  if (!h) return;
  cudaSetDevice(h->cfg.device);
  for (cudaStream_t s : {h->s_main.get(), h->s_index.get(), h->s_copy.get(), h->s_a.get()})
    if (s) cudaStreamSynchronize(s);
  if (h->part)
    for (cudaStream_t s : {h->part->s_pw.get(), h->part->s_pa.get(), h->part->s_pb.get()}) cudaStreamSynchronize(s);
  drain_profile(h);
  delete h;
}

int fi_epp_create(const fi_epp_config* cfg, fi_epp** out) {
  if (!cfg || !out) return FI_ERR_INVALID;
  *out = nullptr;
  std::unique_ptr<fi_epp> up(new fi_epp());
  fi_epp* h = up.get();
  h->cfg = *cfg;
  {
    std::string e;
    int rc = validate_config(*cfg, &e);
    if (rc != FI_OK) {
      std::fprintf(stderr, "fi_epp_create: %s\n", e.c_str());
      return rc;
    }
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    std::fprintf(stderr, "fi_epp_create: no CUDA device — libfi_epp has no CPU fallback\n");
    return FI_ERR_CUDA;
  }
  if (cfg->device < 0 || cfg->device >= ndev) {
    std::fprintf(stderr, "fi_epp_create: device %d out of range (%d devices)\n", cfg->device, ndev);
    return FI_ERR_INVALID;
  }
  auto die = [&](int rc) {
    std::fprintf(stderr, "fi_epp_create: %s\n", h->err.c_str());  // (`up` releases what was created)
    return rc;
  };
#define FI_TRY(call)                                                    \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) {                                           \
      h->err = std::string(#call) + ": " + cudaGetErrorString(e__);     \
      return die(e__ == cudaErrorMemoryAllocation ? FI_ERR_NOMEM : FI_ERR_CUDA); \
    }                                                                   \
  } while (0)
  FI_TRY(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  FI_TRY(cudaGetDeviceProperties(&prop, cfg->device));
  h->sm_count = prop.multiProcessorCount;
  h->P = cfg->n_profiles;
  h->MP = (cfg->max_blocks + 7) & ~7u;  // whole groups of 8 links for the chain walker
  h->W = pow2_ceil32((cfg->endpoint_count + 31) / 32);
  h->fast_hash = (cfg->block_bytes % 32) == 0;
  if (const char* e = std::getenv("FI_EPP_TRACE")) h->trace_call = std::strtol(e, nullptr, 10);
  h->verbose = std::getenv("FI_EPP_VERBOSE") != nullptr;
  if (const char* e = std::getenv("FI_EPP_PIPE_PARTITION")) {
    h->part_want = (int)std::strtol(e, nullptr, 10);
  }
  // (8 ranks on the 8-GPU node ran the partitioned pipeline at 138.5 us per batch with one hashing CTA per request,
  // slower than unpartitioned (133.4 us).  That was first taken for host starvation — 16 cgroup cores for 8 ranks —
  // and the partition switched off there; a single-GPU box then showed the same 138 us with one rank: it is the
  // bimodal co-scheduling that the 4-CTA hashing default removes, so the partition stays on at any rank count.)
  if (const char* e = std::getenv("FI_EPP_WALK_COMPACT")) h->part_compact = std::strtol(e, nullptr, 10) != 0 ? 1 : 0;
  if (const char* e = std::getenv("FI_EPP_PIPE_HASH_CTAS")) h->pipe_hash_ctas = (uint32_t)std::strtol(e, nullptr, 10);
  if (const char* e = std::getenv("FI_EPP_PIPE_MATCH_CTAS")) h->pipe_match_ctas = (uint32_t)std::strtol(e, nullptr, 10);
  if (h->cfg.max_prompt_bytes == 0)
    h->cfg.max_prompt_bytes = (uint64_t)cfg->max_batch * cfg->block_bytes * cfg->max_blocks;
  if (h->cfg.index_slots == 0) {
    // load <= 0.5; an endpoint-range shard is a directory of the WHOLE pool's keys (rows for its own endpoints)
    uint64_t want = 2ull * cfg->num_endpoints * (cfg->lru_capacity ? cfg->lru_capacity : 1024);
    if (want < 4096) want = 4096;
    h->cfg.index_slots = pow2_ceil64(want);
    if (h->cfg.index_slots > 0x80000000ull) h->cfg.index_slots = 0x80000000ull;
  }

  for (Stream* s : {&h->s_main, &h->s_index, &h->s_copy, &h->s_a}) {
    cudaStream_t q = nullptr;
    FI_TRY(cudaStreamCreateWithFlags(&q, cudaStreamNonBlocking));
    s->reset(q);
  }
  for (Event* e : {&h->ev_in, &h->ev_a[0], &h->ev_a[1], &h->ev_b[0], &h->ev_b[1], &h->ev_pick_own, &h->ev_plain})
    FI_TRY(event_create(*e));
  h->ev_pick = h->ev_pick_own.get();
  for (int k = 0; k < fi_epp::kMaxFeedSlices; ++k) FI_TRY(event_create(h->ev_copy[k]));
  if (const char* e = std::getenv("FI_EPP_FEED_SLICES")) {
    const long v = std::strtol(e, nullptr, 10);
    h->feed_slices = (uint32_t)std::min<long>(std::max<long>(v, 1), fi_epp::kMaxFeedSlices);
  }
  for (Event* e : {&h->ev_index, &h->ev_user, &h->ev_done, &h->ev_ctr})
    FI_TRY(event_create(*e));
  FI_TRY(cudaEventRecord(h->ev_index.get(), h->s_index.get()));
  const uint64_t R = cfg->max_batch;
  // rows of the per-request buffers: whole groups of 32 requests (the pre-states are tiled), and — for a shard
  // of a bigger pool — room for the in-place all-gather of `world` equal slices of 32-aligned length
  h->chain_rows = (uint32_t)((R + 31) / 32 * 32);
  if (cfg->endpoint_count < cfg->num_endpoints) h->chain_rows += 32 * (FI_MAX_RANKS + 1);
  if (const char* e = std::getenv("FI_EPP_SHARD_HASH")) h->split_hash = std::strcmp(e, "split") == 0;
  FI_TRY(dev_alloc(h->d_prompts, h->cfg.max_prompt_bytes + 64));
  FI_TRY(dev_alloc(h->d_offsets, (R + 1) * sizeof(uint64_t)));
  FI_TRY(dev_alloc(h->d_h0, R * sizeof(uint64_t)));
  FI_TRY(dev_alloc(h->d_pre, (size_t)h->chain_rows * h->MP * sizeof(uint64_t)));
  FI_TRY(dev_alloc(h->d_chain, (size_t)h->chain_rows * h->MP * sizeof(uint64_t)));
  FI_TRY(dev_alloc(h->d_nblocks, (size_t)h->chain_rows * sizeof(uint32_t)));
  FI_TRY(dev_alloc(h->d_picks, R * h->P * sizeof(fi_pick)));
  FI_TRY(dev_alloc(h->d_probed, 8 * sizeof(unsigned long long)));
  FI_TRY(cudaMemset(h->d_probed.get(), 0, 8 * sizeof(unsigned long long)));
  FI_TRY(dev_alloc(h->d_work, 16 * sizeof(uint32_t)));
  FI_TRY(cudaMemset(h->d_work.get(), 0, 16 * sizeof(uint32_t)));
  FI_TRY(host_alloc(h->h_picks, R * h->P * sizeof(fi_pick)));
  FI_TRY(host_alloc(h->h_offsets, (R + 1) * sizeof(uint64_t)));
  FI_TRY(host_alloc(h->h_h0, R * sizeof(uint64_t)));
  FI_TRY(host_alloc(h->h_nblocks, R * sizeof(uint32_t)));

  // index
  FI_TRY(dev_alloc(h->d_ctr, sizeof(IndexCounters)));
  FI_TRY(cudaMemset(h->d_ctr.get(), 0, sizeof(IndexCounters)));
  FI_TRY(host_alloc(h->h_ctr, sizeof(IndexCounters)));
  std::memset(h->h_ctr.get(), 0, sizeof(IndexCounters));
  {
    int rc = alloc_index(h, h->cfg.index_slots, &h->ix);
    if (rc != FI_OK) return die(rc);
  }
  for (int b = 0; b < 2; ++b) {
    FI_TRY(host_alloc(h->h_sets[b], kOpChunk * sizeof(fi_index_op)));
    FI_TRY(host_alloc(h->h_clears[b], kOpChunk * sizeof(fi_index_op)));
    FI_TRY(dev_alloc(h->d_sets[b], kOpChunk * sizeof(fi_index_op)));
    FI_TRY(dev_alloc(h->d_clears[b], kOpChunk * sizeof(fi_index_op)));
    FI_TRY(event_create(h->ev_buf[b]));
    FI_TRY(cudaEventRecord(h->ev_buf[b].get(), h->s_index.get()));
  }
  if (cfg->lru_capacity) {
    // virtual reservation only: an endpoint's tables become resident when it is first touched
    LruArena* arena = h->lru_arena.reserve((size_t)cfg->endpoint_count * LruSet::bytes_needed(cfg->lru_capacity)) ? &h->lru_arena : nullptr;
    h->lrus = std::vector<LruSet>(cfg->endpoint_count, LruSet(cfg->lru_capacity, arena));
  }

  // endpoints + score tables
  h->eps.assign(cfg->num_endpoints, EndpointDev{0.0, 0, 0, 0, 0});
  const uint32_t Epad = h->W * 32;
  FI_TRY(dev_alloc(h->d_eps, (size_t)cfg->num_endpoints * sizeof(EndpointDev)));
  FI_TRY(dev_alloc(h->d_sc, (size_t)FI_EPP_MAX_PROFILES * FI_EPP_MAX_SCORERS * Epad * sizeof(double)));
  FI_TRY(dev_alloc(h->d_elig, (size_t)FI_EPP_MAX_PROFILES * h->W * sizeof(uint32_t)));
  FI_TRY(dev_alloc(h->d_zero, FI_EPP_MAX_PROFILES * sizeof(ZeroBest)));
  FI_TRY(dev_alloc(h->d_ztie, (size_t)FI_EPP_MAX_PROFILES * h->W * sizeof(uint32_t)));
  FI_TRY(cudaMemset(h->d_ztie.get(), 0, (size_t)FI_EPP_MAX_PROFILES * h->W * sizeof(uint32_t)));
  FI_TRY(cudaMemset(h->d_sc.get(), 0, (size_t)FI_EPP_MAX_PROFILES * FI_EPP_MAX_SCORERS * Epad * sizeof(double)));
  FI_TRY(cudaMemset(h->d_elig.get(), 0, (size_t)FI_EPP_MAX_PROFILES * h->W * sizeof(uint32_t)));
  h->st.n_profiles = h->P;
  h->st.Epad = Epad;
  h->st.sc = h->d_sc.get();
  h->st.elig = h->d_elig.get();
  h->st.zero = h->d_zero.get();
  h->st.ztie = h->d_ztie.get();
  h->lora.assign(Epad, LoraDev{});
  FI_TRY(dev_alloc(h->d_lora, (size_t)Epad * sizeof(LoraDev)));
  FI_TRY(cudaMemset(h->d_lora.get(), 0, (size_t)Epad * sizeof(LoraDev)));
  FI_TRY(dev_alloc(h->d_adapters, R * sizeof(uint64_t)));
  FI_TRY(host_alloc(h->h_adapters, R * sizeof(uint64_t)));
  h->st.lora = h->d_lora.get();
  h->st.has_lora = 0;
  for (uint32_t p = 0; p < h->P; ++p)
    for (uint32_t s = 0; s < cfg->profiles[p].n_scorers; ++s)
      if (cfg->profiles[p].scorers[s].kind == FI_SCORER_LORA) h->st.has_lora = 1;
  for (uint32_t p = 0; p < h->P; ++p) {
    ProfileDev& d = h->st.prof[p];
    d.n_scorers = cfg->profiles[p].n_scorers;
    d.n_filters = 0;
    if (cfg->profiles[p].role_mask) d.filter[d.n_filters++] = cfg->profiles[p].role_mask;
    for (uint32_t f = 0; f < cfg->profiles[p].n_more_filters; ++f) d.filter[d.n_filters++] = cfg->profiles[p].more_filters[f];
    for (uint32_t s = 0; s < d.n_scorers; ++s) {
      d.kind[s] = cfg->profiles[p].scorers[s].kind;
      d.weight[s] = (double)cfg->profiles[p].scorers[s].weight;
    }
  }
  FI_TRY(cudaStreamSynchronize(h->s_index.get()));
  FI_TRY(cudaDeviceSynchronize());
#undef FI_TRY
  *out = up.release();
  return FI_OK;
}

int fi_epp_endpoints_update(fi_epp* h, const fi_endpoint_state* s, uint32_t n) {
  if (!h || (!s && n)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  for (uint32_t i = 0; i < n; ++i) {
    if (s[i].endpoint >= h->cfg.num_endpoints) return fail(h, FI_ERR_INVALID, "endpoint index out of range");
    if (!std::isfinite(s[i].kv_util)) return fail(h, FI_ERR_INVALID, "kv_util must be finite");
  }
  for (uint32_t i = 0; i < n; ++i) {
    EndpointDev& e = h->eps[s[i].endpoint];
    e.kv_util = s[i].kv_util;
    e.queue_depth = s[i].queue_depth;
    e.role_mask = s[i].role_mask;
    e.flags = s[i].flags;
  }
  h->eps_dirty = true;
  return FI_OK;
}

int fi_epp_endpoints_lora_update(fi_epp* h, const fi_endpoint_lora* s, uint32_t n) {
  if (!h || (!s && n)) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  for (uint32_t i = 0; i < n; ++i) {
    if (s[i].endpoint >= h->cfg.num_endpoints) return fail(h, FI_ERR_INVALID, "endpoint index out of range");
    if (s[i].n_active > FI_EPP_MAX_LORA || s[i].n_waiting > FI_EPP_MAX_LORA)
      return fail(h, FI_ERR_INVALID, "more than FI_EPP_MAX_LORA adapters listed");
  }
  for (uint32_t i = 0; i < n; ++i) {
    const uint32_t e = s[i].endpoint - h->cfg.endpoint_begin;
    if (e >= h->cfg.endpoint_count) continue;  // another rank's shard
    LoraDev& d = h->lora[e];
    std::memset(&d, 0, sizeof(d));
    d.n_active = s[i].n_active;
    d.n_waiting = s[i].n_waiting;
    d.max_active = s[i].max_active;
    for (uint32_t k = 0; k < s[i].n_active; ++k) d.active[k] = s[i].active[k];
    for (uint32_t k = 0; k < s[i].n_waiting; ++k) d.waiting[k] = s[i].waiting[k];
  }
  h->lora_dirty = true;
  return FI_OK;
}

int fi_epp_set_option(fi_epp* h, const char* name, int64_t value) {
  if (!h || !name) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  const std::string n(name);
  if (n == "exchange") {
    if (h->world <= 1) return fail(h, FI_ERR_STATE, "exchange: not a sharded pool");
    PeerXchg& px = h->shard->px;
    if (value == FI_EXCHANGE_NCCL) {
      px.enabled = 0;
    } else if (value == FI_EXCHANGE_PEER) {
      if (!px.base[h->rank == 0 ? 1 : 0]) return fail(h, FI_ERR_STATE, "exchange: the peers' buffers were never mapped");
      px.enabled = 1;
    } else {
      return fail(h, FI_ERR_INVALID, "exchange: FI_EXCHANGE_PEER or FI_EXCHANGE_NCCL");
    }
    return FI_OK;
  }
  if (n == "shard_hash") {
    h->split_hash = value != 0;
    return FI_OK;
  }
  if (n == "feed_slices") {
    if (value < 1 || value > fi_epp::kMaxFeedSlices) return fail(h, FI_ERR_INVALID, "feed_slices: 1..16");
    h->feed_slices = (uint32_t)value;
    return FI_OK;
  }
  if (n == "pipe_hash_ctas" || n == "pipe_match_ctas") {
    if (value < 0 || value > 4096) return fail(h, FI_ERR_INVALID, n + ": 0..4096");
    (n == "pipe_hash_ctas" ? h->pipe_hash_ctas : h->pipe_match_ctas) = (uint32_t)value;
    return FI_OK;
  }
  if (n == "device_lru") {
    if (value != 0 && value != 1) return fail(h, FI_ERR_INVALID, "device_lru: 0 or 1");
    if (h->lru_mode >= 0 && h->lru_mode != (int)value) return fail(h, FI_ERR_STATE, "device_lru: the handle's LRU is already in use");
    h->lru_want = (int)value;
    return FI_OK;
  }
  if (n == "pipe_partition") {
    if (value < 0 || value > 64) return fail(h, FI_ERR_INVALID, "pipe_partition: 0 (off) or the walker partition's SM count");
    if (h->part && value == 0) {
      // back to the unpartitioned pipeline, and the partition is released; nothing of the partitioned pipeline may
      // still be in flight: the two share the pre-state / chain buffers
      cudaSetDevice(h->cfg.device);
      for (cudaStream_t st : {h->part->s_pa.get(), h->part->s_pw.get(), h->part->s_pb.get()}) cudaStreamSynchronize(st);
      h->ev_pick = h->ev_pick_own.get();  // (it may name a slot event of the partition; those picks are done)
      h->part.reset();
      h->part_active = false;
    } else if (!h->part) {
      h->part_want = (int)value;
      h->part_tried = false;
    }
    return FI_OK;
  }
  if (n == "lru_table_slots") {
    if (value < 0 || value > (1ll << 30)) return fail(h, FI_ERR_INVALID, "lru_table_slots: 0 .. 2^30");
    if (h->dlru) return fail(h, FI_ERR_STATE, "lru_table_slots: the device LRU is already allocated");
    h->lru_table_slots = (uint32_t)value;
    return FI_OK;
  }
  if (n == "lru_threads") {
    if (value < 1 || value > 1024) return fail(h, FI_ERR_INVALID, "lru_threads: 1..1024");
    h->lru_threads = (unsigned)value;
    h->pool.reset();
    return FI_OK;
  }
  return fail(h, FI_ERR_INVALID, "unknown option: " + n);
}

int fi_epp_set_profiling(fi_epp* h, int on) {
  if (!h) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  cudaSetDevice(h->cfg.device);
  drain_profile(h);
  h->profiling = on != 0;
  return FI_OK;
}

int fi_epp_get_stats(fi_epp* h, fi_epp_stats* out) {
  if (!h || !out) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) return fail(h, FI_ERR_CUDA, "cudaSetDevice failed");
  drain_profile(h);
  if (h->profiling) {
    FI_CUDA(cudaStreamSynchronize(h->s_main.get()));
    unsigned long long pb[8] = {0};
    FI_CUDA(cudaMemcpy(pb, h->d_probed.get(), sizeof(pb), cudaMemcpyDeviceToHost));
    h->stats.probed_blocks = pb[0];
    if (pb[5] && h->verbose)  // FI_MATCH_TIMING build: where a request's time goes inside match_pick
      std::fprintf(stderr, "[fi_epp] match_pick phases, cycles per request over %llu requests: stage %.0f, first lookup %.0f, "
                   "chunks %.0f, score+pick %.0f\n", pb[5], (double)pb[1] / pb[5], (double)pb[2] / pb[5], (double)pb[3] / pb[5],
                   (double)pb[4] / pb[5]);
  }
  *out = h->stats;
  return FI_OK;
}

int fi_epp_reset_stats(fi_epp* h) {
  if (!h) return FI_ERR_INVALID;
  std::lock_guard<std::mutex> lk(h->mu);
  cudaSetDevice(h->cfg.device);
  drain_profile(h);
  cudaStreamSynchronize(h->s_main.get());
  cudaMemset(h->d_probed.get(), 0, 8 * sizeof(unsigned long long));
  h->stats = fi_epp_stats{};
  return FI_OK;
}

}  // extern "C"
