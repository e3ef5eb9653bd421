// lru_kernels.cu — the per-endpoint LRU of block hashes, resident on the GPU (sm_100a).
//
// Upstream keeps one LRU per pod (podToLRU, SURVEY.md Appendix A.2; capacity lruCapacityPerServer,
// /root/reference/pkg/router/strategy.go:59,149) and runs indexer.Add(chain, pod) for every routed request.
// On a host that is a pointer chase per block — a few DRAM misses each, ~95 M touches/s on the 16 usable
// cores of the GPU box, 330 K decisions/s at 256 blocks per prompt — three orders of magnitude below the pick
// rate.  Here the recency order lives in HBM next to the index and a whole batch of Adds is applied by a handful
// of wide kernels; only the request → endpoint assignment (two small arrays) comes from the host.
//
// Exactness.  An LRU of capacity C always holds the C most recently touched distinct keys, whatever it evicted
// on the way.  So the state after a batch of touches depends only on every key's LAST touch: per endpoint, the
// keys touched in the batch, ordered by their last touch (the WINNERS), go behind everything older, and the
// content is cut to the newest C.  A winner followed by C or more other winners is gone again by the end of the
// batch (DOOMED: CLEARed — sequential Adds would have SET and evicted it, so the pair ends up absent whatever put
// it into the index before); the index gets SET for the surviving winners that were new to the endpoint and CLEAR
// for the entries that fell off — the same membership as R sequential Adds, whatever those inserted and evicted
// in between.
//
// Capacity.  A table takes the batch's distinct keys on top of its C entries; it holds 0.85 TS, with TS between
// 4 C and 32 C slots depending on how much HBM is free (engine_lru.cu: a B200 gives 1 024 endpoints 1 Mi slots each).
// An endpoint that receives more NEW distinct keys than that in a single batch is detected while inserting
// (slots are reserved before they are claimed), its touches are rolled back and its requests are re-run in
// sub-batches of at most C touches, which always fit (lru_plan.h; endpoints are independent of each other, so
// deferring one is exact).
//
// Per endpoint e (all in HBM):
//   table  [TS + 2] LruSlot   open-addressed, linear probing, key → (log position + 1, order of its last touch
//                             in the running sub-batch).  Slots TS / TS+1 belong to the hashes 0 / ~0 (the
//                             table's EMPTY / TOMB markers).  Evicted entries become tombstones; a rehash
//                             (maintenance) drops them.
//   log    [L] u64            the recency order: one record per (key, touch that was the key's last in its
//                             sub-batch), appended in touch order.  A record is LIVE iff the table still
//                             points at it; everything else is a stale leftover of an older touch.  The live
//                             records between tail and head, oldest first, ARE the LRU list.
//   head, tail, count (live entries), used (table slots consumed)
//
// One sub-batch = kernels  maintain → touch → (untouch) → count → scan → append → [index SET] → evict → [index CLEAR]:
//   maintain  endpoints whose log could overflow: compact it (live records only, renumbered from 0; the table
//             follows); endpoints whose table is crowded with tombstones: rebuild it from the compacted log
//                                                                                    one CTA per endpoint
//   touch     find-or-insert every (endpoint, key); atomicMax of the touch order    one CTA per request
//   untouch   (only after an overflow) undo the touches of the overflowed endpoints
//   count     a touch is a WINNER iff it is its key's last touch of the sub-batch; winners per request
//   scan      per endpoint, requests in order: log position of each request's first winner; new head
//   append    surviving winners write their log record, point the table at it, emit SET if the key was new;
//             doomed winners leave the table (CLEAR if they were entries before)
//   evict     endpoints above capacity: walk the log from the tail, evict the oldest live records, emit CLEAR
#include "kernels.cuh"
#include "lru_device.cuh"

namespace fi {

namespace {

constexpr uint32_t LRU_MISS = 0xFFFFFFFFu;
// the per-endpoint kernels (evict, maintain) walk an endpoint's log with ONE CTA, a block of records per step with
// a dependent table lookup each: the widest CTA keeps a hot endpoint's walk (up to `capacity` evictions) short
constexpr int kWideCta = 1024;

__device__ __forceinline__ uint32_t lru_home(uint64_t key, uint32_t mask) {
  // the index table buckets by the low bits of the hash: use high ones here
  return (uint32_t)((key * 0x9E3779B97F4A7C15ull) >> 40) & mask;
}

__device__ __forceinline__ unsigned long long vload64(const uint64_t* p) {
  return *reinterpret_cast<const volatile unsigned long long*>(p);
}

// slot of `key` in endpoint table `tab`, inserting it if absent (*inserted).  A new key first reserves one of
// the table's insert_limit slots (`used`); LRU_MISS when there is none left (the caller flags the overflow).
__device__ uint32_t lru_find_or_insert(LruSlot* tab, uint32_t TS, uint64_t key, uint32_t* used, uint32_t limit, bool* inserted) {
  *inserted = false;
  if (key == KEY_EMPTY || key == KEY_TOMB) {
    const uint32_t s = TS + (key == KEY_TOMB ? 1u : 0u);
    const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&tab[s].key), 0ull, 1ull);
    *inserted = old == 0ull;
    return s;
  }
  const uint32_t mask = TS - 1;
  uint32_t i = lru_home(key, mask);
  bool reserved = false;
  for (uint32_t it = 0; it < TS; ++it) {
    const unsigned long long k = vload64(&tab[i].key);
    if (k == key) {
      if (reserved) atomicSub(used, 1u);  // someone else inserted it meanwhile
      return i;
    }
    if (k == KEY_EMPTY) {
      if (!reserved) {
        if (atomicAdd(used, 1u) >= limit) {
          atomicSub(used, 1u);
          return LRU_MISS;
        }
        reserved = true;
      }
      const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&tab[i].key), 0ull, (unsigned long long)key);
      if (old == 0ull) {
        *inserted = true;
        return i;
      }
      if (old == key) {
        atomicSub(used, 1u);
        return i;
      }
    }
    i = (i + 1) & mask;
  }
  if (reserved) atomicSub(used, 1u);
  return LRU_MISS;
}

__device__ uint32_t lru_find(const LruSlot* tab, uint32_t TS, uint64_t key) {
  if (key == KEY_EMPTY || key == KEY_TOMB) {
    const uint32_t s = TS + (key == KEY_TOMB ? 1u : 0u);
    return tab[s].key ? s : LRU_MISS;
  }
  const uint32_t mask = TS - 1;
  uint32_t i = lru_home(key, mask);
  for (uint32_t it = 0; it < TS; ++it) {
    const uint64_t k = tab[i].key;
    if (k == key) return i;
    if (k == KEY_EMPTY) return LRU_MISS;
    i = (i + 1) & mask;
  }
  return LRU_MISS;
}

__device__ __forceinline__ void lru_retire(LruSlot* tab, uint32_t TS, uint32_t slot) {
  tab[slot].posp1 = 0;
  tab[slot].ord = 0;
  tab[slot].key = slot >= TS ? 0ull : KEY_TOMB;  // the two special slots are simply freed
}

// CTA-wide exclusive scan of a flag (any whole number of warps up to 32); returns this thread's rank,
// *total = number of flags set
__device__ uint32_t cta_rank(bool flag, uint32_t* total) {
  __shared__ uint32_t s_w[32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  const unsigned m = __ballot_sync(0xFFFFFFFFu, flag);
  if (lane == 0) s_w[warp] = __popc(m);
  __syncthreads();
  // every warp scans the (at most 32) warp totals with its own lanes
  const uint32_t c = lane < nw ? s_w[lane] : 0u;
  uint32_t inc = c;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
    if ((int)lane >= d) inc += t;
  }
  const uint32_t tot = __shfl_sync(0xFFFFFFFFu, inc, 31);
  const uint32_t before = __shfl_sync(0xFFFFFFFFu, inc - c, warp);
  __syncthreads();  // s_w is reused by the next call
  *total = tot;
  return before + __popc(m & ((1u << lane) - 1u));
}

// ---- touch ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lru_touch_kernel(DevLru lru, LruBatch b) {
  const uint32_t k = blockIdx.x;
  const uint32_t e = b.req_ep[k], n = b.req_n[k], off = b.req_off[k];
  LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  const uint64_t* chain = b.chains + (uint64_t)b.req_id[k] * b.pitch;
  for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
    const uint64_t key = chain[j];
    bool ins = false;
    const uint32_t slot = lru_find_or_insert(tab, lru.TS, key, lru.used + e, lru.insert_limit, &ins);
    b.slot_of[off + j] = slot;
    if (slot == LRU_MISS) {  // the table cannot take this batch's distinct keys: the endpoint is deferred
      lru.ovf[e] = 1u;
      *lru.any_ovf = 1u;
      continue;
    }
    atomicMax(&tab[slot].ord, off + j + 1);
  }
}

// ---- untouch: roll back the touches of the endpoints that overflowed -----------------------------------
__global__ void __launch_bounds__(256) lru_untouch_kernel(DevLru lru, LruBatch b) {
  const uint32_t k = blockIdx.x;
  const uint32_t e = b.req_ep[k], n = b.req_n[k], off = b.req_off[k];
  if (!lru.ovf[e]) return;
  LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) {
    const uint32_t slot = b.slot_of[off + j];
    if (slot == LRU_MISS) continue;
    // keys this sub-batch inserted have no log record yet: they leave again (as tombstones: the re-run's
    // maintenance pass rebuilds the table); entries that were there before just forget the touch.  Several
    // touches of one key write the same values.
    if (tab[slot].posp1 == 0) lru_retire(tab, lru.TS, slot);
    else tab[slot].ord = 0;
  }
}

// ---- count ----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lru_count_kernel(DevLru lru, LruBatch b) {
  const uint32_t k = blockIdx.x;
  const uint32_t e = b.req_ep[k], n = b.req_n[k], off = b.req_off[k];
  const LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  uint32_t wins = 0;
  const bool deferred = lru.ovf[e] != 0;
  for (uint32_t j = threadIdx.x; j < n && !deferred; j += blockDim.x) {
    const uint32_t slot = b.slot_of[off + j];
    if (slot != LRU_MISS && tab[slot].ord == off + j + 1) ++wins;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) wins += __shfl_xor_sync(0xFFFFFFFFu, wins, d);
  __shared__ uint32_t s_tot;
  if (threadIdx.x == 0) s_tot = 0;
  __syncthreads();
  if ((threadIdx.x & 31) == 0 && wins) atomicAdd(&s_tot, wins);
  __syncthreads();
  if (threadIdx.x == 0) b.wcount[k] = s_tot;
}

// ---- scan: one warp per endpoint, its requests in order ----------------------------------------------
__global__ void __launch_bounds__(256) lru_scan_kernel(DevLru lru, LruBatch b) {
  const uint32_t e = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (e >= lru.EL) return;
  const uint32_t i0 = b.ep_start[e], i1 = b.ep_start[e + 1];
  if (i0 == i1) return;
  uint32_t running = 0;
  for (uint32_t i = i0; i < i1; i += 32) {
    const bool v = i + lane < i1;
    const uint32_t k = v ? b.ep_list[i + lane] : 0;
    const uint32_t w = v ? b.wcount[k] : 0;
    uint32_t inc = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t t = __shfl_up_sync(0xFFFFFFFFu, inc, d);
      if ((int)lane >= d) inc += t;
    }
    if (v) b.base[k] = running + inc - w;
    running += __shfl_sync(0xFFFFFFFFu, inc, 31);
  }
  if (lane == 0) {
    const uint32_t head = lru.head[e];
    const uint32_t kept = running < lru.capacity ? running : lru.capacity;  // the doomed winners get no record
    lru.hold[e] = head;
    lru.dcount[e] = running;
    if ((uint64_t)head + kept > lru.L) atomicExch(lru.error, 2u);  // cannot happen: maintenance runs first
    lru.head[e] = head + kept;
  }
}

// ---- append -----------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lru_append_kernel(DevLru lru, LruBatch b, fi_index_op* clears, unsigned long long* n_clears,
                                                         uint64_t clears_cap, uint32_t ep_begin) {
  const uint32_t k = blockIdx.x;
  const uint32_t e = b.req_ep[k], n = b.req_n[k], off = b.req_off[k];
  LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  uint64_t* log = lru.log + (uint64_t)e * lru.L;
  const uint64_t* chain = b.chains + (uint64_t)b.req_id[k] * b.pitch;
  const bool deferred = lru.ovf[e] != 0;
  const uint32_t D = lru.dcount[e], hold = lru.hold[e];
  const uint32_t doomed_below = D > lru.capacity ? D - lru.capacity : 0;  // winners of rank < this are gone again
  uint32_t at = b.base[k];  // rank of this request's next winner among the endpoint's winners
  uint32_t fresh = 0, lost = 0, doomed = 0;
  for (uint32_t j0 = 0; j0 < n; j0 += blockDim.x) {  // uniform trip count: block-wide barriers inside
    const uint32_t j = j0 + threadIdx.x;
    uint32_t slot = LRU_MISS;
    bool win = false;
    if (j < n && !deferred) {
      slot = b.slot_of[off + j];
      win = slot != LRU_MISS && tab[slot].ord == off + j + 1;
    }
    uint32_t tot = 0;
    const uint32_t rank = at + cta_rank(win, &tot);
    fi_index_op op{0, 0, 0};
    if (win) {
      const uint64_t key = chain[j];
      const bool was_entry = tab[slot].posp1 != 0;
      if (rank < doomed_below) {
        // touched, but C or more distinct keys were touched after it: not in the LRU at the end of the batch.
        // Sequential Adds would have SET it and evicted (CLEARed) it again, so the pair must end up absent from
        // the index even if something else put it there (fi_epp_index_apply bypasses the LRU): always CLEAR
        lru_retire(tab, lru.TS, slot);
        ++doomed;
        if (was_entry) ++lost;
        const unsigned long long c = atomicAdd(n_clears, 1ull);
        if (c < clears_cap) clears[c] = fi_index_op{key, ep_begin + e, FI_OP_CLEAR};
      } else {
        const uint32_t p = hold + (rank - doomed_below);
        if (p < lru.L) log[p] = key;
        if (!was_entry) {  // new to this endpoint
          op = fi_index_op{key, ep_begin + e, FI_OP_SET};
          ++fresh;
        }
        tab[slot].posp1 = p + 1;
        tab[slot].ord = 0;
      }
    }
    if (j < n) b.sets[off + j] = op;
    at += tot;
  }
  // per-CTA totals: entries gained / lost
  __shared__ uint32_t s_fresh, s_lost, s_doomed;
  if (threadIdx.x == 0) s_fresh = s_lost = s_doomed = 0;
  __syncthreads();
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    fresh += __shfl_xor_sync(0xFFFFFFFFu, fresh, d);
    lost += __shfl_xor_sync(0xFFFFFFFFu, lost, d);
    doomed += __shfl_xor_sync(0xFFFFFFFFu, doomed, d);
  }
  if ((threadIdx.x & 31) == 0) {
    if (fresh) atomicAdd(&s_fresh, fresh);
    if (lost) atomicAdd(&s_lost, lost);
    if (doomed) atomicAdd(&s_doomed, doomed);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_fresh) {
      atomicAdd(lru.count + e, s_fresh);
      atomicAdd(lru.n_sets, (unsigned long long)s_fresh);
    }
    if (s_lost) atomicSub(lru.count + e, s_lost);
    if (s_doomed) {
      atomicAdd(lru.n_doomed, (unsigned long long)s_doomed);
      atomicAdd(lru.n_clears, (unsigned long long)s_doomed);
    }
  }
}

// ---- evict: one CTA per endpoint above capacity ------------------------------------------------------
__global__ void __launch_bounds__(kWideCta) lru_evict_kernel(DevLru lru, fi_index_op* clears, unsigned long long* n_clears,
                                                        uint64_t clears_cap, uint32_t ep_begin) {
  const uint32_t e = blockIdx.x;
  const uint32_t cnt = lru.count[e];
  if (cnt <= lru.capacity) return;
  uint32_t need = cnt - lru.capacity;
  LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  const uint64_t* log = lru.log + (uint64_t)e * lru.L;
  const uint32_t head = lru.head[e];
  uint32_t t = lru.tail[e];
  while (need > 0 && t < head) {
    const uint32_t p = t + threadIdx.x;
    uint64_t key = 0;
    uint32_t slot = LRU_MISS;
    bool live = false;
    if (p < head) {
      key = log[p];
      slot = lru_find(tab, lru.TS, key);
      live = slot != LRU_MISS && tab[slot].posp1 == p + 1;
    }
    uint32_t tot = 0;
    const uint32_t rank = cta_rank(live, &tot);
    const bool go = live && rank < need;
    if (go) {
      lru_retire(tab, lru.TS, slot);
      const unsigned long long at = atomicAdd(n_clears, 1ull);
      if (at < clears_cap) clears[at] = fi_index_op{key, ep_begin + e, FI_OP_CLEAR};
    }
    if (tot >= need) {
      // the record of the last eviction ends the walk: the tail moves right behind it
      __shared__ uint32_t s_last;
      if (go && rank == need - 1) s_last = p;
      __syncthreads();
      t = s_last + 1;
      need = 0;
    } else {
      need -= tot;
      t += blockDim.x;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    if (need) atomicExch(lru.error, 3u);  // fewer live records than entries: cannot happen
    lru.tail[e] = t < head ? t : head;
    lru.count[e] = lru.capacity + need;
    atomicAdd(lru.n_clears, (unsigned long long)(cnt - lru.capacity - need));
  }
}

// ---- maintain: compact the log, rebuild the table -------------------------------------------------------
__global__ void __launch_bounds__(kWideCta) lru_maintain_kernel(DevLru lru, const uint32_t* __restrict__ inc, uint32_t force) {
  const uint32_t e = blockIdx.x;
  const uint32_t add = inc ? inc[e] : 0;
  const uint32_t head = lru.head[e];
  // the log takes at most `capacity` more records per sub-batch (doomed winners get none); the table should
  // stay at most 60 % full if the sub-batch brings the usual amount of new keys (more is caught by the insert limit)
  const uint32_t addc = add < lru.capacity ? add : lru.capacity;
  const bool log_tight = (uint64_t)head + addc > lru.L;
  const bool tab_tight = ((uint64_t)lru.used[e] + addc) * 10 > (uint64_t)lru.TS * 6;
  if (!force && !log_tight && !tab_tight) return;
  LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  uint64_t* log = lru.log + (uint64_t)e * lru.L;
  // 1. live records move to the front, in order, and the table follows them (a chunk is read completely before
  //    any of it is rewritten, and the write cursor never passes the read cursor; a key's stale records all lie
  //    before its live one, so a rewritten position is never mistaken for one of them)
  uint32_t d = 0;
  for (uint32_t t = lru.tail[e]; t < head; t += blockDim.x) {
    const uint32_t p = t + threadIdx.x;
    uint64_t key = 0;
    uint32_t slot = LRU_MISS;
    bool live = false;
    if (p < head) {
      key = log[p];
      slot = lru_find(tab, lru.TS, key);
      live = slot != LRU_MISS && tab[slot].posp1 == p + 1;
    }
    uint32_t tot = 0;
    const uint32_t rank = cta_rank(live, &tot);  // (barriers inside: reads above are done)
    if (live) {
      log[d + rank] = key;
      tab[slot].posp1 = d + rank + 1;
    }
    d += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    lru.tail[e] = 0;
    lru.head[e] = d;
    if (d != lru.count[e]) atomicExch(lru.error, 5u);  // live records == entries, always
    atomicAdd(lru.n_maintained, 1ull);
  }
  if (!force && !tab_tight) return;
  // 2. tombstones crowd the table: a fresh one from the compacted log (the two special slots keep their place)
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (uint32_t i = threadIdx.x; i < lru.TS; i += blockDim.x) reinterpret_cast<uint4*>(tab)[i] = z;
  if (threadIdx.x == 0) lru.used[e] = 0;
  __syncthreads();
  uint32_t regular = 0;
  for (uint32_t i = threadIdx.x; i < d; i += blockDim.x) {
    const uint64_t key = log[i];
    if (key == KEY_EMPTY || key == KEY_TOMB) continue;
    bool ins = false;
    const uint32_t slot = lru_find_or_insert(tab, lru.TS, key, lru.used + e, lru.TS, &ins);
    if (slot == LRU_MISS) {
      atomicExch(lru.error, 4u);
      continue;
    }
    tab[slot].posp1 = i + 1;
    ++regular;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) regular += __shfl_xor_sync(0xFFFFFFFFu, regular, s);
  __shared__ uint32_t s_tot;
  if (threadIdx.x == 0) s_tot = 0;
  __syncthreads();
  if ((threadIdx.x & 31) == 0 && regular) atomicAdd(&s_tot, regular);
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(lru.used + e, 0u) != s_tot) atomicExch(lru.error, 6u);
}

// diagnostics (tests): the live keys of endpoint e, oldest first
__global__ void __launch_bounds__(256) lru_dump_kernel(DevLru lru, uint32_t e, uint64_t* out, uint32_t* n_out) {
  const LruSlot* tab = lru.slots + (uint64_t)e * (lru.TS + 2);
  const uint64_t* log = lru.log + (uint64_t)e * lru.L;
  const uint32_t head = lru.head[e];
  uint32_t d = 0;
  for (uint32_t t = lru.tail[e]; t < head; t += blockDim.x) {
    const uint32_t p = t + threadIdx.x;
    uint64_t key = 0;
    bool live = false;
    if (p < head) {
      key = log[p];
      const uint32_t slot = lru_find(tab, lru.TS, key);
      live = slot != LRU_MISS && tab[slot].posp1 == p + 1;
    }
    uint32_t tot = 0;
    const uint32_t rank = cta_rank(live, &tot);
    if (live) out[d + rank] = key;
    d += tot;
  }
  if (threadIdx.x == 0) *n_out = d;
}

}  // namespace

cudaError_t launch_lru_maintain(const DevLru& lru, const uint32_t* inc, bool force, cudaStream_t s) {
  lru_maintain_kernel<<<lru.EL, kWideCta, 0, s>>>(lru, inc, force ? 1u : 0u);
  return cudaGetLastError();
}
cudaError_t launch_lru_touch(const DevLru& lru, const LruBatch& b, cudaStream_t s) {
  if (b.K == 0) return cudaSuccess;
  lru_touch_kernel<<<b.K, 256, 0, s>>>(lru, b);
  return cudaGetLastError();
}
cudaError_t launch_lru_untouch(const DevLru& lru, const LruBatch& b, cudaStream_t s) {
  if (b.K == 0) return cudaSuccess;
  lru_untouch_kernel<<<b.K, 256, 0, s>>>(lru, b);
  return cudaGetLastError();
}
cudaError_t launch_lru_count(const DevLru& lru, const LruBatch& b, cudaStream_t s) {
  if (b.K == 0) return cudaSuccess;
  lru_count_kernel<<<b.K, 256, 0, s>>>(lru, b);
  return cudaGetLastError();
}
cudaError_t launch_lru_scan(const DevLru& lru, const LruBatch& b, cudaStream_t s) {
  lru_scan_kernel<<<(lru.EL + 7) / 8, 256, 0, s>>>(lru, b);
  return cudaGetLastError();
}
cudaError_t launch_lru_append(const DevLru& lru, const LruBatch& b, fi_index_op* clears, unsigned long long* n_clears,
                              uint64_t clears_cap, uint32_t ep_begin, cudaStream_t s) {
  if (b.K == 0) return cudaSuccess;
  lru_append_kernel<<<b.K, 256, 0, s>>>(lru, b, clears, n_clears, clears_cap, ep_begin);
  return cudaGetLastError();
}
cudaError_t launch_lru_evict(const DevLru& lru, fi_index_op* clears, unsigned long long* n_clears, uint64_t clears_cap,
                             uint32_t ep_begin, cudaStream_t s) {
  lru_evict_kernel<<<lru.EL, kWideCta, 0, s>>>(lru, clears, n_clears, clears_cap, ep_begin);
  return cudaGetLastError();
}
cudaError_t launch_lru_dump(const DevLru& lru, uint32_t e, uint64_t* out, uint32_t* n_out, cudaStream_t s) {
  lru_dump_kernel<<<1, 256, 0, s>>>(lru, e, out, n_out);
  return cudaGetLastError();
}

}  // namespace fi
