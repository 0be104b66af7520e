// index.cu — kvblock index (request key -> pod entries) and longest-prefix scorer, DEVICE-AUTHORITATIVE.
//
// Replaces InMemoryIndex (pkg/kvcache/kvblock/in_memory.go:57-304) and
// LongestPrefixScorer.Score (pkg/kvcache/kvblock_scorer.go:91-154).
//
// Where the state lives
//   * request key -> pod entries: an open-addressing table of 64 B buckets {key, state|count, 13 x (pod:16|tier:8|spec:8)}
//     in HBM, plus one 64-bit recency stamp per slot (ts[]).  There is NO host copy: Add / Evict are applied to the
//     buckets by kernels, Lookup / Score read them, and the outer LRU of the reference (golang-lru, `Size` keys) is the
//     order of the stamps — every operation that golang-lru would move to the front (`data.Get` in Lookup, Add and
//     Evict) stamps the slot with a global sequence number handed out in the reference's operation order.
//   * engine key -> request keys (in_memory.go:166-177): a flat hash map with an intrusive LRU list on the host; it is
//     touched once per engine key of an event, never by reads.
// Mutations
//   Add / Evict append 16 B op records to a pinned queue and return.  A flush (before the next read, or when the queue
//   is full) ships the queue and applies it in one of two ways:
//     parallel   sort ops by key (stable, cub radix sort), one thread per DISTINCT key replays that key's ops in order
//                on the bucket held in registers (the 13-entry inner LRU is a register loop) and writes it back once;
//                used whenever no outer-LRU eviction can happen (live + new <= Size);
//     sequential one thread replays the queue in order, evicting the oldest key exactly when the reference would
//                (contains_or_add past `Size`).  "Oldest" comes from an order array (stamp, slot) sorted once on the
//                device and consumed lazily: a record is stale when its slot was re-stamped or freed.  Exact LRU at
//                capacity, amortised O(1) per eviction; also used for tiny batches (one launch, no sort).
//   The table grows by a device-side rehash; nothing is ever rebuilt from the host.
// Reads
//   Lookup: one thread per key.  Score: one warp per prompt — 32 independent probes staged in shared memory, then the
//   serial float64 prefix walk in key order (bit-identical sums, kvblock_scorer.go:132-150).  Found keys are stamped
//   by the kernel (atomicMax), so refreshing recency costs the host nothing.
// Random-access bound (2 sectors per probe), not bandwidth bound.
//
// The same source compiles with g++ -DKVB_HOST_SIM against tests/cpp/sim_cuda.h (malloc + loops instead of a device) so
// the mutation logic is checked against the oracle on CPU-only boxes; the product build has no such path.
#ifdef KVB_HOST_SIM
#include "sim_cuda.h"
#define KVB_DEV
#else
#define KVB_DEV __device__
#include <cub/cub.cuh>

#include "kvb_internal.h"
#define KVB_LAUNCH(kernel, grid, block, stream, ...) kernel<<<(grid), (block), 0, (stream)>>>(__VA_ARGS__)
#endif

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "index_device.cuh"

namespace kvb {

constexpr uint8_t kOpAdd = 0, kOpEvict = 1;
struct OpRec {  // one queued mutation of one request key
  uint64_t key;
  uint32_t ent_off;  // first entry in the entry pool
  uint16_t ent_cnt;
  uint8_t type;
  uint8_t pad;
};
static_assert(sizeof(OpRec) == 16, "op record must be 16 B");

struct Counters {  // device resident
  unsigned long long live, tombs, order_head, evicted, inserted, removed, stale_skipped, scans;
  long long resume_at;            // sequential replay: first op not yet applied, -1 when the batch is done
  unsigned long long pending_evict;  // an eviction the replay still owes (its order array ran out)
  unsigned long long purge_entries, purge_keys;  // pod removal: entries removed / keys deleted by the last sweep
};

struct TableRef {
  Bucket* table;
  unsigned long long* ts;
  uint64_t mask;
  Counters* ctr;
  int ppk;
};

KVB_DEV __forceinline__ uint32_t ld_meta(const Bucket* b) {
  return *reinterpret_cast<const volatile uint32_t*>(&b->meta);
}
KVB_DEV __forceinline__ uint64_t ld_key(const Bucket* b) {
  return *reinterpret_cast<const volatile uint64_t*>(&b->key);
}

// slot of `key` or -1; *reuse = first free (empty or tombstone) slot on the probe path, -1 if the table is full
KVB_DEV inline int64_t find_slot(const TableRef& t, uint64_t key, int64_t* reuse) {
  uint64_t slot = mix64(key) & t.mask;
  int64_t free_slot = -1;
  for (uint64_t probes = 0; probes <= t.mask; ++probes, slot = (slot + 1) & t.mask) {
    const uint32_t st = ld_meta(&t.table[slot]) & 3u;
    if (st == kEmpty) {
      if (free_slot < 0) free_slot = (int64_t)slot;
      break;
    }
    if (st == kTomb) {
      if (free_slot < 0) free_slot = (int64_t)slot;
    } else if (st == kFull && ld_key(&t.table[slot]) == key) {
      if (reuse) *reuse = free_slot;
      return (int64_t)slot;
    }
  }
  if (reuse) *reuse = free_slot;
  return -1;
}

// claim a free slot for a NEW key (threads of one launch carry distinct keys, so a lost race just moves on);
// the slot is left in state kBusy for the caller to fill.  Returns -1 only if the table has no free slot.
KVB_DEV inline int64_t claim_slot(const TableRef& t, uint64_t key, int64_t hint, bool* was_tomb) {
  uint64_t slot = hint >= 0 ? (uint64_t)hint : (mix64(key) & t.mask);
  for (uint64_t probes = 0; probes <= t.mask; ++probes, slot = (slot + 1) & t.mask) {
    const uint32_t m = ld_meta(&t.table[slot]);
    const uint32_t st = m & 3u;
    if (st != kEmpty && st != kTomb) continue;
    if (atomicCAS(&t.table[slot].meta, m, kBusy) != m) {
      --probes;  // somebody else moved this slot: look at it again
      slot = (slot - 1) & t.mask;
      continue;
    }
    *was_tomb = st == kTomb;
    return (int64_t)slot;
  }
  return -1;
}

// inner LRU of one key (golang-lru Add on PodEntry, oldest first): an entry already present moves to newest, a new
// one evicts the oldest when the key already holds `ppk` entries (in_memory.go:205-221, in_memory_test.go:86-120)
KVB_DEV inline void inner_add(uint32_t* ent, int& cnt, uint32_t e, int ppk) {
  int at = -1;
  for (int k = 0; k < cnt; ++k)
    if (ent[k] == e) {
      at = k;
      break;
    }
  if (at >= 0) {
    for (int k = at; k + 1 < cnt; ++k) ent[k] = ent[k + 1];
    ent[cnt - 1] = e;
    return;
  }
  if (cnt == ppk) {
    for (int k = 0; k + 1 < cnt; ++k) ent[k] = ent[k + 1];
    --cnt;
  }
  ent[cnt++] = e;
}
KVB_DEV inline void inner_remove(uint32_t* ent, int& cnt, uint32_t e) {  // exact triple match (:266-269)
  for (int k = 0; k < cnt; ++k)
    if (ent[k] == e) {
      for (int q = k; q + 1 < cnt; ++q) ent[q] = ent[q + 1];
      --cnt;
      return;
    }
}

KVB_DEV inline void store_bucket(const TableRef& t, int64_t slot, uint64_t key, const uint32_t* ent,
                                              int cnt, bool fresh) {
  Bucket& b = t.table[slot];
  if (fresh) b.key = key;
  for (int e = 0; e < kMaxEnt; ++e) b.ent[e] = e < cnt ? ent[e] : 0u;
  __threadfence();
  *reinterpret_cast<volatile uint32_t*>(&b.meta) = kFull | ((uint32_t)cnt << 8);
}
KVB_DEV inline void kill_slot(const TableRef& t, int64_t slot) {
  *reinterpret_cast<volatile uint32_t*>(&t.table[slot].meta) = kTomb;
  t.ts[slot] = 0ull;
}

// ---- parallel path: thread i owns the run of ops that carry sorted key skey[i] (only the run's first thread works)
KVB_DEV inline void apply_run(const TableRef& t, const OpRec* ops, const uint32_t* ents,
                                          const uint64_t* skey, const uint32_t* sidx, int64_t i, int64_t n,
                                          unsigned long long seq_base) {
  const uint64_t key = skey[i];
  if (i > 0 && skey[i - 1] == key) return;
  int64_t reuse = -1;
  const int64_t found = find_slot(t, key, &reuse);
  uint32_t ent[kMaxEnt];
  int cnt = 0;
  bool present = found >= 0;
  if (present) {
    const Bucket& b = t.table[found];
    cnt = (int)((ld_meta(&b) >> 8) & 0xffu);
    for (int e = 0; e < kMaxEnt; ++e) ent[e] = b.ent[e];
  }
  unsigned long long stamp = 0ull;
  for (int64_t j = i; j < n && skey[j] == key; ++j) {
    const OpRec op = ops[sidx[j]];
    if (op.type == kOpAdd) {
      if (!present) {  // data.Get missed: a fresh inner LRU (in_memory.go:186-199)
        present = true;
        cnt = 0;
      }
      stamp = seq_base + sidx[j];
      for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_add(ent, cnt, ents[op.ent_off + e], t.ppk);
    } else if (present) {  // evictPodsFromRequestKey: Get refreshes recency, then removes (in_memory.go:260-292)
      stamp = seq_base + sidx[j];
      for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_remove(ent, cnt, ents[op.ent_off + e]);
      if (cnt == 0) present = false;
    }
  }
  if (found >= 0) {
    if (present) {
      store_bucket(t, found, key, ent, cnt, false);
      if (stamp) t.ts[found] = stamp;
    } else {
      kill_slot(t, found);
      atomicAdd(&t.ctr->live, (unsigned long long)-1ll);
      atomicAdd(&t.ctr->tombs, 1ull);
      atomicAdd(&t.ctr->removed, 1ull);
    }
  } else if (present) {
    bool was_tomb = false;
    const int64_t s = claim_slot(t, key, reuse, &was_tomb);
    if (s < 0) return;  // cannot happen: the host grows the table before it fills
    store_bucket(t, s, key, ent, cnt, true);
    t.ts[s] = stamp;
    atomicAdd(&t.ctr->live, 1ull);
    atomicAdd(&t.ctr->inserted, 1ull);
    if (was_tomb) atomicAdd(&t.ctr->tombs, (unsigned long long)-1ll);
  }
}

// ---- sequential path (one thread): the reference's order, including outer-LRU eviction at `max_keys`
// false: the order array ran out and the table is too large to scan for the minimum — the caller stops, the host
// rebuilds the order array and resumes (a scan per eviction is fine for a few thousand slots, not for 10^8)
KVB_DEV inline bool evict_oldest(const TableRef& t, const unsigned long long* order_ts,
                                             const uint32_t* order_slot, unsigned long long order_n,
                                             unsigned long long scan_max_slots) {
  Counters& c = *t.ctr;
  while (c.order_head < order_n) {  // lazily validated order array
    const unsigned long long h = c.order_head++;
    const uint32_t s = order_slot[h];
    if ((ld_meta(&t.table[s]) & 3u) == kFull && t.ts[s] == order_ts[h]) {
      kill_slot(t, s);
      c.live--;
      c.tombs++;
      c.evicted++;
      return true;
    }
    c.stale_skipped++;
  }
  // order exhausted (more insertions than the array held, or lookups re-stamped what was left): the keys left are newer
  // than every record
  if (t.mask + 1 > scan_max_slots) return false;
  c.scans++;
  int64_t best = -1;
  unsigned long long best_ts = ~0ull;
  for (uint64_t s = 0; s <= t.mask; ++s)
    if ((ld_meta(&t.table[s]) & 3u) == kFull && t.ts[s] < best_ts) {
      best_ts = t.ts[s];
      best = (int64_t)s;
    }
  if (best >= 0) {
    kill_slot(t, best);
    c.live--;
    c.tombs++;
    c.evicted++;
  }
  return true;
}

KVB_DEV inline void apply_seq(const TableRef& t, const OpRec* ops, const uint32_t* ents, int64_t start, int64_t n,
                                          unsigned long long seq_base, unsigned long long max_keys,
                                          const unsigned long long* order_ts, const uint32_t* order_slot,
                                          unsigned long long order_n, unsigned long long scan_max_slots) {
  Counters& c = *t.ctr;
  if (c.pending_evict) {  // resumed after the order array was rebuilt: the eviction the previous launch still owed
    c.pending_evict = 0;
    evict_oldest(t, order_ts, order_slot, order_n, ~0ull);
  }
  c.resume_at = -1;
  for (int64_t j = start; j < n; ++j) {
#ifndef KVB_HOST_SIM
    constexpr int64_t kAhead = 12;  // the one thread walks dependent DRAM probes: pull the home buckets of the next ops into L2
    if (j + kAhead < n) {
      const Bucket* nb = &t.table[mix64(ops[j + kAhead].key) & t.mask];
      asm volatile("prefetch.global.L2 [%0];" ::"l"(nb));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(&t.ts[mix64(ops[j + kAhead].key) & t.mask]));
    }
#endif
    const OpRec op = ops[j];
    int64_t reuse = -1;
    int64_t slot = find_slot(t, op.key, &reuse);
    uint32_t ent[kMaxEnt] = {};
    int cnt = 0;
    if (op.type == kOpAdd) {
      bool fresh = false;
      if (slot < 0) {
        bool was_tomb = false;
        slot = claim_slot(t, op.key, reuse, &was_tomb);
        if (slot < 0) return;
        fresh = true;
        c.live++;
        c.inserted++;
        if (was_tomb) c.tombs--;
        store_bucket(t, slot, op.key, ent, 0, true);
        t.ts[slot] = seq_base + j;  // newest before the eviction looks for the oldest
        if (c.live > max_keys && !evict_oldest(t, order_ts, order_slot, order_n, scan_max_slots)) {  // lru.Add past Size (in_memory.go:197)
          // out of order records on a large table: finish this op, then hand back to the host for a fresh order array
          for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_add(ent, cnt, ents[op.ent_off + e], t.ppk);
          store_bucket(t, slot, op.key, ent, cnt, true);
          c.pending_evict = 1;
          c.resume_at = j + 1;
          return;
        }
      } else {
        const Bucket& b = t.table[slot];
        cnt = (int)((ld_meta(&b) >> 8) & 0xffu);
        for (int e = 0; e < kMaxEnt; ++e) ent[e] = b.ent[e];
        t.ts[slot] = seq_base + j;
      }
      for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_add(ent, cnt, ents[op.ent_off + e], t.ppk);
      store_bucket(t, slot, op.key, ent, cnt, fresh);
    } else if (slot >= 0) {
      const Bucket& b = t.table[slot];
      cnt = (int)((ld_meta(&b) >> 8) & 0xffu);
      for (int e = 0; e < kMaxEnt; ++e) ent[e] = b.ent[e];
      for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_remove(ent, cnt, ents[op.ent_off + e]);
      if (cnt == 0) {
        kill_slot(t, slot);
        c.live--;
        c.tombs++;
        c.removed++;
      } else {
        store_bucket(t, slot, op.key, ent, cnt, false);
        t.ts[slot] = seq_base + j;
      }
    }
  }
}

// ----------------------------------------------------------------------------------------- kernels
__global__ void index_apply_par_kernel(TableRef t, const OpRec* __restrict__ ops, const uint32_t* __restrict__ ents,
                                       const uint64_t* __restrict__ skey, const uint32_t* __restrict__ sidx, int64_t n,
                                       unsigned long long seq_base) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  apply_run(t, ops, ents, skey, sidx, i, n, seq_base);
}

__global__ void index_apply_seq_kernel(TableRef t, const OpRec* __restrict__ ops, const uint32_t* __restrict__ ents,
                                       int64_t start, int64_t n, unsigned long long seq_base,
                                       unsigned long long max_keys, const unsigned long long* __restrict__ order_ts,
                                       const uint32_t* __restrict__ order_slot, unsigned long long order_n,
                                       unsigned long long scan_max_slots) {
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  apply_seq(t, ops, ents, start, n, seq_base, max_keys, order_ts, order_slot, order_n, scan_max_slots);
}

// ---- pod removal (kvb_index_remove_pods): one sweep over every slot.  No reference counterpart: the reference ignores
// AllBlocksCleared (pool.go:388-395) and only removes a pod through Evict of keys the caller names.
struct TierMask {  // 256 device tiers, one bit each; travels in the kernel arguments
  uint32_t bits[8];
};

// One bucket: drop every entry whose pod is in `pod_bits` and whose tier is in `tiers` (the speculative bit is not
// looked at), keep the rest in their inner-LRU order and write the bucket back only if it changed.  A key left empty is
// deleted, as evictPodsFromRequestKey does (in_memory.go:281-292).  The recency stamp of a surviving key is NOT touched.
// Returns the entries removed; *deleted = the key was deleted.
KVB_DEV inline uint32_t purge_bucket(const TableRef& t, int64_t slot, uint32_t meta, const uint32_t* ent,
                                     const uint32_t* __restrict__ pod_bits, const TierMask& tiers, bool* deleted) {
  *deleted = false;
  if ((meta & 3u) != kFull) return 0u;
  const int raw_cnt = (int)((meta >> 8) & 0xffu), cnt = raw_cnt < kMaxEnt ? raw_cnt : kMaxEnt;
  uint32_t keep[kMaxEnt];
  int n = 0;
#pragma unroll
  for (int e = 0; e < kMaxEnt; ++e) keep[e] = 0u;
#pragma unroll
  for (int e = 0; e < kMaxEnt; ++e) {
    if (e >= cnt) break;
    const uint32_t v = ent[e], pod = v & 0xffffu, tier = (v >> 16) & 0xffu;
    if (((pod_bits[pod >> 5] >> (pod & 31u)) & 1u) && ((tiers.bits[tier >> 5] >> (tier & 31u)) & 1u)) continue;
#pragma unroll
    for (int j = 0; j <= e; ++j)  // static indices: keep[] stays in registers
      if (j == n) keep[j] = v;
    ++n;
  }
  if (n == cnt) return 0u;
  if (n == 0) {
    kill_slot(t, slot);
    *deleted = true;
  } else {
    store_bucket(t, slot, 0ull, keep, n, false);
  }
  return (uint32_t)(cnt - n);
}

KVB_DEV __forceinline__ void load_bucket(const Bucket* b, uint32_t* meta, uint32_t* ent) {
#ifndef KVB_HOST_SIM
  const uint4* src = reinterpret_cast<const uint4*>(b);  // key | meta ent0 | ent1-4 | ent5-8 | ent9-12
  const uint4 q0 = src[0], q1 = src[1], q2 = src[2], q3 = src[3];
  *meta = q0.z;
  ent[0] = q0.w;
  ent[1] = q1.x, ent[2] = q1.y, ent[3] = q1.z, ent[4] = q1.w;
  ent[5] = q2.x, ent[6] = q2.y, ent[7] = q2.z, ent[8] = q2.w;
  ent[9] = q3.x, ent[10] = q3.y, ent[11] = q3.z, ent[12] = q3.w;
#else
  *meta = b->meta;
  for (int e = 0; e < kMaxEnt; ++e) ent[e] = b->ent[e];
#endif
}

// Persistent grid, grid-stride over the slots, kPurgeUnroll buckets per thread per step: their 64 B loads are all issued
// before any is looked at, so every thread keeps 128 B in flight.  Counters are summed per warp and added once per warp.
constexpr int kPurgeThreads = 256, kPurgeUnroll = 2;

__global__ void __launch_bounds__(kPurgeThreads)
    index_remove_pods_kernel(TableRef t, const uint32_t* __restrict__ pod_bits, TierMask tiers) {
  const uint64_t n_slots = t.mask + 1;
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  uint32_t removed = 0u, deleted = 0u;
  for (uint64_t s0 = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s0 < n_slots; s0 += stride * kPurgeUnroll) {
    uint32_t meta[kPurgeUnroll], ent[kPurgeUnroll][kMaxEnt];
#pragma unroll
    for (int u = 0; u < kPurgeUnroll; ++u) {
      const uint64_t s = s0 + (uint64_t)u * stride;
      meta[u] = kEmpty;
      if (s < n_slots) load_bucket(&t.table[s], &meta[u], ent[u]);
    }
#pragma unroll
    for (int u = 0; u < kPurgeUnroll; ++u) {
      bool del = false;
      removed += purge_bucket(t, (int64_t)(s0 + (uint64_t)u * stride), meta[u], ent[u], pod_bits, tiers, &del);
      deleted += del ? 1u : 0u;
    }
  }
#ifndef KVB_HOST_SIM
  removed = __reduce_add_sync(0xffffffffu, removed);
  deleted = __reduce_add_sync(0xffffffffu, deleted);
  if ((threadIdx.x & 31) != 0) return;
#endif
  if (removed == 0u) return;
  Counters& c = *t.ctr;
  atomicAdd(&c.purge_entries, (unsigned long long)removed);
  if (deleted == 0u) return;
  atomicAdd(&c.purge_keys, (unsigned long long)deleted);
  atomicAdd(&c.live, (unsigned long long)(-(long long)deleted));
  atomicAdd(&c.tombs, (unsigned long long)deleted);
  atomicAdd(&c.removed, (unsigned long long)deleted);
}

__global__ void index_sort_keys_kernel(const OpRec* __restrict__ ops, int64_t n, uint64_t* __restrict__ keys,
                                       uint32_t* __restrict__ idx) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  keys[i] = ops[i].key;
  idx[i] = (uint32_t)i;
}

// move every live bucket (and its stamp) into a larger table
__global__ void index_rehash_kernel(const Bucket* __restrict__ old_table, const unsigned long long* __restrict__ old_ts,
                                    uint64_t old_slots, TableRef t) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= old_slots) return;
  const Bucket& b = old_table[s];
  if ((b.meta & 3u) != kFull) return;
  bool was_tomb = false;
  const int64_t d = claim_slot(t, b.key, -1, &was_tomb);
  if (d < 0) return;
  store_bucket(t, d, b.key, b.ent, (int)((b.meta >> 8) & 0xffu), true);
  t.ts[d] = old_ts[s];
}

// (stamp, slot) of every live bucket, in arbitrary order (sorted afterwards)
__global__ void index_collect_order_kernel(TableRef t, unsigned long long* __restrict__ out_ts,
                                           uint32_t* __restrict__ out_slot, unsigned long long* __restrict__ cursor,
                                           unsigned long long cap) {
  const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (s > t.mask) return;
  if ((t.table[s].meta & 3u) != kFull) return;
  const unsigned long long at = atomicAdd(cursor, 1ull);
  if (at < cap) {
    out_ts[at] = t.ts[s];
    out_slot[at] = (uint32_t)s;
  }
}

// ---- parallel apply AT CAPACITY.  The reference evicts the outer LRU's oldest key at every insertion that pushes the
// cache past Size (lru.Add, in_memory.go:197), one op at a time.  The same victims can be planned before anything is
// applied.  Replaying each key's ops on its own (the sorted runs) tells which ops INSERT a key (+1) and which DELETE one
// (its last pod leaves: -1); with net_t = live + the sum of those events up to op t, eviction number e happens at the
// first op whose net reaches Size + e + 1 — evictions only ever trim the excess, so their count after op t is the
// running maximum of net minus Size.  Its victim is the e-th record of the recency order that the batch has not touched
// by then.  A record the batch touches BEFORE the eviction that would reach it has moved to the newest end and survives;
// one it touches only AFTER is evicted and its later ops act on an absent key — a "conflict" key: a victim, and a
// different event sequence (an insertion where there was a touch), which shifts the plan.  So the conflict set is
// recomputed from scratch until the plan reproduces itself.  Victims are removed before the apply kernel runs, so a
// conflict key is simply absent when its ops are replayed.
//
// events: the run head replays its key's ops on a register copy of the bucket (nothing is written to the table)
__global__ void index_plan_events_kernel(TableRef t, const OpRec* __restrict__ ops, const uint32_t* __restrict__ ents,
                                         const uint64_t* __restrict__ skey, const uint32_t* __restrict__ sidx, int64_t n,
                                         const uint8_t* __restrict__ conflict, int32_t* __restrict__ ev) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t key = skey[i];
  if (i > 0 && skey[i - 1] == key) return;
  const int64_t found = conflict[i] ? -1 : find_slot(t, key, nullptr);  // a conflict key is gone before its first op
  uint32_t ent[kMaxEnt];
  int cnt = 0;
  bool present = found >= 0;
  if (present) {
    const Bucket& b = t.table[found];
    cnt = (int)((ld_meta(&b) >> 8) & 0xffu);
    for (int e = 0; e < kMaxEnt; ++e) ent[e] = b.ent[e];
  }
  for (int64_t j = i; j < n && skey[j] == key; ++j) {
    const OpRec op = ops[sidx[j]];
    if (op.type == kOpAdd) {
      if (!present) {
        present = true;
        cnt = 0;
        ev[sidx[j]] = 1;
      }
      for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_add(ent, cnt, ents[op.ent_off + e], t.ppk);
    } else if (present) {
      for (uint32_t e = 0; e < op.ent_cnt; ++e) inner_remove(ent, cnt, ents[op.ent_off + e]);
      if (cnt == 0) {
        present = false;
        ev[sidx[j]] = -1;
      }
    }
  }
}

// net[t] = events up to and including op t, top[t] = their running maximum.  An insertion that lifts live to a new
// maximum above Size is the op of eviction number (that maximum - Size - 1).
__global__ void index_evict_times_kernel(const int32_t* __restrict__ ev, const int32_t* __restrict__ net,
                                         const int32_t* __restrict__ top, int64_t n, int64_t live0, int64_t max_keys,
                                         uint32_t* __restrict__ evict_op) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || ev[i] <= 0) return;
  const int64_t cur = live0 + net[i];
  const int64_t prev_top = i > 0 ? (int64_t)top[i - 1] : 0;
  const int64_t before = live0 + (prev_top > 0 ? prev_top : 0);
  if (cur > max_keys && cur > before) evict_op[cur - max_keys - 1] = (uint32_t)i;
}

constexpr uint32_t kUntouched = 0xffffffffu;

// one window of the order array.  touch[p] = position of the record's key among the sorted batch keys (its run head:
// the stable sort puts the key's first op there) or kUntouched; is_victim[p] = valid record that is untouched or a
// known conflict key.  Stale records (re-stamped or removed since the order was built) are neither.
__global__ void index_evict_flag_kernel(TableRef t, const unsigned long long* __restrict__ order_ts,
                                        const uint32_t* __restrict__ order_slot, int64_t pos, int64_t w,
                                        const uint64_t* __restrict__ skey, int64_t n, const uint8_t* __restrict__ conflict,
                                        uint32_t* __restrict__ is_victim, uint32_t* __restrict__ touch) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= w) return;
  const uint32_t s = order_slot[pos + p];
  uint32_t vic = 0, tch = kUntouched;
  if ((ld_meta(&t.table[s]) & 3u) == kFull && t.ts[s] == order_ts[pos + p]) {
    const uint64_t key = ld_key(&t.table[s]);
    int64_t lo = 0, hi = n;  // first position with skey >= key
    while (lo < hi) {
      const int64_t mid = (lo + hi) >> 1;
      if (skey[mid] < key) lo = mid + 1;
      else hi = mid;
    }
    if (lo < n && skey[lo] == key) {
      tch = (uint32_t)lo;
      vic = conflict[lo];
    } else {
      vic = 1;
    }
  }
  is_victim[p] = vic;
  touch[p] = tch;
}

// rank[p] = victims (under the current conflict set) before p in this window; `found` were taken from earlier
// windows, `need` more are wanted.  Every touched record is decided afresh into conflict_next.
// out[0] = records whose decision differs from the current set, out[1] = window position just past the last victim
// taken, out[2] = victims taken here, out[3] = size of the next conflict set
__global__ void index_evict_decide_kernel(const uint32_t* __restrict__ is_victim, const uint32_t* __restrict__ touch,
                                          const uint32_t* __restrict__ rank, int64_t w, int64_t pos,
                                          const uint32_t* __restrict__ order_slot, const uint32_t* __restrict__ sidx,
                                          int64_t found, int64_t need, const uint32_t* __restrict__ evict_op,
                                          uint8_t* __restrict__ conflict_next, uint32_t* __restrict__ victims,
                                          unsigned long long* __restrict__ out) {
  const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= w) return;
  const int64_t r = (int64_t)rank[p];
  const uint32_t tch = touch[p];
  const bool vic = is_victim[p] != 0;
  if (r >= need) {  // past the last eviction of this batch: not looked at, so a conflict key out here stops being one
    if (vic && tch != kUntouched) atomicAdd(&out[0], 1ull);
    return;
  }
  if (tch != kUntouched) {
    const bool c = sidx[tch] > evict_op[found + r];  // first touched only after the eviction reaches it
    if (c) {
      conflict_next[tch] = 1;
      atomicAdd(&out[3], 1ull);
    }
    if (c != vic) atomicAdd(&out[0], 1ull);
  }
  if (vic) {
    victims[found + r] = order_slot[pos + p];
    if (r == need - 1) out[1] = (unsigned long long)(p + 1);
    atomicAdd(&out[2], 1ull);
  }
}

__global__ void index_evict_apply_kernel(TableRef t, const uint32_t* __restrict__ victims, int64_t n_victims,
                                         unsigned long long new_head, unsigned long long skipped) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_victims) return;
  kill_slot(t, victims[i]);
  if (i == 0) {
    Counters& c = *t.ctr;
    atomicAdd(&c.live, (unsigned long long)(-(long long)n_victims));
    atomicAdd(&c.tombs, (unsigned long long)n_victims);
    atomicAdd(&c.evicted, (unsigned long long)n_victims);
    atomicAdd(&c.stale_skipped, skipped);
    c.order_head = new_head;
  }
}

// Lookup: one thread per key.  counts: -1 absent, -2 present but empty, else #entries after the pod filter.
// stamp_base != 0: found keys are re-stamped (data.Get, in_memory.go:120) with stamp_base + position.
__global__ void index_lookup_kernel(const Bucket* __restrict__ table, uint64_t mask, const uint64_t* __restrict__ keys,
                                    int64_t n, const uint32_t* __restrict__ filter_bits, int32_t* __restrict__ counts,
                                    uint32_t* __restrict__ out_ent, unsigned long long* __restrict__ ts,
                                    unsigned long long stamp_base) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t s = probe(table, mask, keys[i]);
  if (s < 0) {
    counts[i] = -1;
    return;
  }
  if (stamp_base) atomicMax(&ts[s], stamp_base + (unsigned long long)i);
  const Bucket& b = table[s];
  const int cnt = (int)((b.meta >> 8) & 0xff);
  if (cnt == 0) {
    counts[i] = -2;
    return;
  }
  int k = 0;
  for (int e = 0; e < cnt; ++e) {
    const uint32_t v = b.ent[e];
    if (pod_allowed(filter_bits, v & 0xffffu)) out_ent[i * kMaxEnt + k++] = v;
  }
  counts[i] = k;
}

#ifndef KVB_HOST_SIM
// Score: one warp per prompt (4 warps per CTA); the walk itself is ScoreWalker (index_device.cuh), shared with the
// fused tokens -> scores kernel of hash_kernels.cu.
constexpr int kScoreWarps = 4;

__global__ void __launch_bounds__(kScoreWarps * 32)
    index_score_kernel(const Bucket* __restrict__ table, uint64_t mask, const uint64_t* __restrict__ keys,
                       const int64_t* __restrict__ key_off, int32_t n_prompts,
                       const uint32_t* __restrict__ filter_bits, const double* __restrict__ tier_w,
                       int32_t* __restrict__ out_n, uint16_t* __restrict__ out_pods, double* __restrict__ out_scores,
                       unsigned long long* __restrict__ ts /* nullable: stamp found keys */,
                       unsigned long long stamp_base) {
  __shared__ Bucket tile[kScoreWarps][32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int p = blockIdx.x * kScoreWarps + warp;
  if (p >= n_prompts) return;
  const int64_t k0 = key_off[p];
  const int64_t nk = key_off[p + 1] - k0;
  ScoreWalker wk;
  for (int64_t base = 0; base < nk; base += 32) {
    if (!wk.chain_alive && ts == nullptr) break;
    const int64_t ki = base + lane;
    const uint64_t key = ki < nk ? keys[k0 + ki] : 0ull;
    wk.tile(table, mask, tile[warp], key, ki < nk, base, (int)min((int64_t)32, nk - base), filter_bits, tier_w, ts,
            stamp_base + (unsigned long long)(k0 + ki));
  }
  wk.finish(p, out_n, out_pods, out_scores);
}
#endif  // !KVB_HOST_SIM

// ----------------------------------------------------------------------------------------- host side
// engine key -> request keys with golang-lru semantics (Add: update + move to newest, evict oldest past `cap`;
// Get: move to newest).  Flat: nodes in a vector linked by index, open-addressing index with backward-shift delete.
class EngMap {
 public:
  static constexpr uint32_t kNil = 0xffffffffu;
  struct Node {
    uint64_t ek = 0, rk_last = 0;
    uint32_t n = 0, prev = kNil, next = kNil;
    std::vector<uint64_t>* many = nullptr;  // all request keys when n > 1
  };
  explicit EngMap(int64_t cap) : cap_(cap) { rebuild(1024); }
  ~EngMap() {
    for (auto& nd : nodes_) delete nd.many;
  }
  size_t size() const { return size_; }
  int64_t find(uint64_t ek) const {
    for (size_t i = home(ek);; i = (i + 1) & mask_) {
      const uint32_t v = tab_[i];
      if (v == 0) return -1;
      if (nodes_[v - 1].ek == ek) return (int64_t)(v - 1);
    }
  }
  const Node& node(int64_t id) const { return nodes_[(size_t)id]; }
  void touch(int64_t id) {
    unlink((uint32_t)id);
    push_back((uint32_t)id);
  }
  void put(uint64_t ek, const uint64_t* rks, size_t n) {
    int64_t id = find(ek);
    if (id >= 0) {
      set_value(nodes_[(size_t)id], rks, n);
      touch(id);
      return;
    }
    uint32_t nid;
    if (!free_.empty()) {
      nid = free_.back();
      free_.pop_back();
    } else {
      nid = (uint32_t)nodes_.size();
      nodes_.emplace_back();
    }
    if ((size_ + 1) * 2 > tab_.size()) rebuild(tab_.size() * 2);  // before the node joins the list rebuild() walks
    Node& nd = nodes_[nid];
    nd.ek = ek;
    set_value(nd, rks, n);
    push_back(nid);
    insert_index(nid);
    ++size_;
    if ((int64_t)size_ > cap_ && head_ != kNil) erase(head_);
  }
  void erase(int64_t id) {
    const Node& nd = nodes_[(size_t)id];
    size_t i = home(nd.ek);
    while (tab_[i] != (uint32_t)id + 1) i = (i + 1) & mask_;
    for (;;) {  // backward-shift deletion
      tab_[i] = 0;
      size_t j = i;
      for (;;) {
        j = (j + 1) & mask_;
        if (tab_[j] == 0) goto done;
        const size_t k = home(nodes_[tab_[j] - 1].ek);
        const bool stays = (i <= j) ? (i < k && k <= j) : (i < k || k <= j);
        if (!stays) break;
      }
      tab_[i] = tab_[j];
      i = j;
    }
  done:
    unlink((uint32_t)id);
    delete nodes_[(size_t)id].many;
    nodes_[(size_t)id] = Node();
    free_.push_back((uint32_t)id);
    --size_;
  }
  template <class F>
  void for_each_rk(int64_t id, F&& f) const {
    const Node& nd = nodes_[(size_t)id];
    if (nd.n == 1) f(nd.rk_last);
    else if (nd.many)
      for (uint64_t rk : *nd.many) f(rk);
  }

 private:
  int64_t cap_;
  std::vector<Node> nodes_;
  std::vector<uint32_t> free_;
  std::vector<uint32_t> tab_;
  size_t mask_ = 0, size_ = 0;
  uint32_t head_ = kNil, tail_ = kNil;  // head = oldest

  size_t home(uint64_t ek) const { return (size_t)mix64(ek) & mask_; }
  static void set_value(Node& nd, const uint64_t* rks, size_t n) {
    nd.n = (uint32_t)n;
    nd.rk_last = n ? rks[n - 1] : 0;
    if (n > 1) {
      if (!nd.many) nd.many = new std::vector<uint64_t>();
      nd.many->assign(rks, rks + n);
    } else {
      delete nd.many;
      nd.many = nullptr;
    }
  }
  void insert_index(uint32_t nid) {
    size_t i = home(nodes_[nid].ek);
    while (tab_[i] != 0) i = (i + 1) & mask_;
    tab_[i] = nid + 1;
  }
  void rebuild(size_t cap) {
    tab_.assign(cap, 0u);
    mask_ = cap - 1;
    for (uint32_t id = head_; id != kNil; id = nodes_[id].next) insert_index(id);
  }
  void unlink(uint32_t id) {
    Node& nd = nodes_[id];
    if (nd.prev != kNil) nodes_[nd.prev].next = nd.next;
    else if (head_ == id) head_ = nd.next;
    if (nd.next != kNil) nodes_[nd.next].prev = nd.prev;
    else if (tail_ == id) tail_ = nd.prev;
    nd.prev = nd.next = kNil;
  }
  void push_back(uint32_t id) {
    Node& nd = nodes_[id];
    nd.prev = tail_;
    nd.next = kNil;
    if (tail_ != kNil) nodes_[tail_].next = id;
    tail_ = id;
    if (head_ == kNil) head_ = id;
  }
};

}  // namespace kvb

using namespace kvb;

struct kvb_index {
  int device = 0;
  int64_t max_keys = 0;
  int pods_per_key = 10;
  std::mutex mu;
  std::unique_ptr<EngMap> eng;

  // device table
  Bucket* table = nullptr;
  unsigned long long* ts = nullptr;
  uint64_t slots = 0;
  Counters* d_ctr = nullptr;
  Counters h_ctr{};        // last value read back
  int64_t live_ub = 0;     // upper bound on live keys, including queued adds
  int64_t tomb_ub = 0;     // upper bound on tombstones
  unsigned long long seq = 1;  // next recency stamp (0 = never stamped)
  cudaStream_t stream = nullptr;
  double tier_w_host[256];
  double* tier_w = nullptr;

  // pinned op queue + device copies and sort buffers
  static constexpr size_t kOpsCap = 1u << 18, kEntsCap = 1u << 20;
  static constexpr int64_t kSeqThreshold = 16;  // batches this small skip the sort and replay on one thread
  OpRec* h_ops = nullptr;
  uint32_t* h_ents = nullptr;
  size_t n_ops = 0, n_ents = 0;
  int64_t q_adds = 0, q_evicts = 0;
  cudaEvent_t q_free = nullptr;  // the previous flush's H2D copies have read the pinned queue
  bool q_busy = false;
  OpRec* d_ops = nullptr;
  uint32_t* d_ents = nullptr;
  uint64_t *d_skey_in = nullptr, *d_skey_out = nullptr;
  uint32_t *d_sidx_in = nullptr, *d_sidx_out = nullptr;
  void* d_sort_tmp = nullptr;
  size_t sort_tmp_bytes = 0;

  // LRU order array (built on demand, only when the index runs at capacity)
  unsigned long long* order_ts = nullptr;
  uint32_t* order_slot = nullptr;
  unsigned long long *order_ts_in = nullptr, *d_cursor = nullptr;
  uint32_t* order_slot_in = nullptr;
  int64_t order_cap = 0, order_n = 0;
  bool order_valid = false;
  // eviction planner (parallel apply at capacity): one window of the order array at a time
  static constexpr int64_t kWinCap = 1 << 20;
  uint32_t *d_plan_ops = nullptr, *d_victims = nullptr, *d_win = nullptr;  // d_plan_ops: ev | net | top | evict_op; d_win: is_victim | touch | rank
  unsigned long long* d_plan = nullptr;                                     // see index_evict_decide_kernel
  uint8_t* d_conflict = nullptr;                                            // per sorted batch position

  // read scratch
  uint8_t* d_scratch = nullptr;
  size_t d_scratch_cap = 0;
  uint8_t* h_scratch = nullptr;
  uint8_t* h_scratch_dev = nullptr;  // device alias of the pinned staging block (taken once, when it is allocated)
  size_t h_scratch_cap = 0;
  uint32_t* d_filter = nullptr;  // 65536 bits
  uint32_t* d_purge_bits = nullptr;  // 65536 bits: the pods of the running kvb_index_remove_pods
  unsigned* d_done = nullptr;                 // prompts finished in the running fused launch (the kernel resets it)
  unsigned long long* h_done = nullptr;       // pinned word the last prompt writes the call's sequence number to
  unsigned long long done_seq = 0;
  std::vector<uint16_t> filter_cached;
  bool filter_valid = false;
  cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_c = nullptr;
  float last_hash_us = 0.f, last_score_us = 0.f;
#ifndef KVB_HOST_SIM
  SpecScratch* spec = nullptr;  // tables of the table kernel (small scoring batches, small ingest rounds)
#endif

  // statistics
  int64_t n_flush_par = 0, n_flush_seq = 0, n_rehash = 0, n_order_builds = 0, n_ops_total = 0;
  int64_t n_flush_planned = 0, n_plan_fallbacks = 0, n_seq_resumes = 0;

  TableRef ref() const { return TableRef{table, ts, slots - 1, d_ctr, pods_per_key}; }

  int ensure_scratch(size_t dev_bytes, size_t host_bytes) {
    if (dev_bytes > d_scratch_cap) {
      if (d_scratch) cudaFree(d_scratch);
      d_scratch = nullptr;
      d_scratch_cap = 0;  // a failed allocation below must not leave a stale capacity behind
      size_t cap = std::max<size_t>(dev_bytes, 1 << 20);
      cap = (cap * 3 / 2 + 255) & ~size_t(255);
      KVB_CUDA_TRY(cudaMalloc(&d_scratch, cap));
      d_scratch_cap = cap;
    }
    if (host_bytes > h_scratch_cap) {
      if (h_scratch) cudaFreeHost(h_scratch);
      h_scratch = nullptr;
      h_scratch_cap = 0;
      size_t cap = std::max<size_t>(host_bytes, 1 << 20);
      cap = (cap * 3 / 2 + 255) & ~size_t(255);
      KVB_CUDA_TRY(host_alloc_near(device, reinterpret_cast<void**>(&h_scratch), cap,
                                   cudaHostAllocPortable | cudaHostAllocMapped));
      h_scratch_cap = cap;
      h_scratch_dev = h_scratch;  // UVA: pinned host memory is addressable by kernels at the same address ...
#ifndef KVB_HOST_SIM
      void* alias = nullptr;    // ... and the runtime confirms it where it can
      if (cudaHostGetDevicePointer(&alias, h_scratch, 0) == cudaSuccess && alias) h_scratch_dev = static_cast<uint8_t*>(alias);
      else cudaGetLastError();
#endif
    }
    return KVB_OK;
  }

  int alloc_table(uint64_t n_slots, Bucket** t_out, unsigned long long** ts_out) {
    Bucket* t = nullptr;
    unsigned long long* s = nullptr;
    KVB_CUDA_TRY(cudaMalloc(&t, n_slots * sizeof(Bucket)));
    if (cudaMalloc(&s, n_slots * sizeof(unsigned long long)) != cudaSuccess) {
      cudaFree(t);
      set_error("index: cannot allocate %llu recency stamps", (unsigned long long)n_slots);
      return KVB_ERR_CUDA;
    }
    cudaError_t e = cudaMemsetAsync(t, 0, n_slots * sizeof(Bucket), stream);
    if (e == cudaSuccess) e = cudaMemsetAsync(s, 0, n_slots * sizeof(unsigned long long), stream);
    if (e != cudaSuccess) {
      cudaFree(t);
      cudaFree(s);
      set_error("index: clearing a new table failed: %s", cudaGetErrorString(e));
      return KVB_ERR_CUDA;
    }
    *t_out = t;
    *ts_out = s;
    return KVB_OK;
  }

  int sync_counters() {  // exact live / tombstone counts (waits for everything queued on the stream)
    KVB_CUDA_TRY(cudaMemcpyAsync(&h_ctr, d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, stream));
    KVB_CUDA_TRY(cudaStreamSynchronize(stream));
    live_ub = (int64_t)h_ctr.live + q_adds;
    tomb_ub = (int64_t)h_ctr.tombs + q_evicts;
    return KVB_OK;
  }

  int rehash(uint64_t new_slots);
  int ensure_order(int64_t min_records = 1);
  int ensure_sort_tmp(size_t need);
  int plan_evictions(int64_t n, int64_t* n_victims, unsigned long long* new_head, unsigned long long* skipped, bool* ok);
  int flush_locked();
  int flush_piece(size_t first, size_t count, bool may_evict);
  int queue_ops(uint8_t type, const uint64_t* keys, int64_t n_keys, const kvb_pod_entry_t* entries, int32_t n_entries);
  int set_filter(const uint16_t* pods, int32_t n, uint8_t* h_stage, bool* staged, const uint32_t** out);
  int remove_pods_locked(const uint16_t* pods, int32_t n_pods, const uint8_t* tiers, int32_t n_tiers,
                         int64_t* entries_removed, int64_t* keys_deleted);
};

int kvb_index::rehash(uint64_t new_slots) {
  Bucket* fresh = nullptr;
  unsigned long long* fresh_ts = nullptr;
  int rc = alloc_table(new_slots, &fresh, &fresh_ts);  // a failed allocation leaves the index as it was
  if (rc) return rc;
  TableRef nt{fresh, fresh_ts, new_slots - 1, d_ctr, pods_per_key};
  const unsigned threads = 256;
  KVB_LAUNCH(index_rehash_kernel, (unsigned)((slots + threads - 1) / threads), threads, stream, table, ts, slots, nt);
  KVB_CUDA_TRY(cudaGetLastError());
  count_launch();
  Counters zero_tombs;
  KVB_CUDA_TRY(cudaMemcpyAsync(&zero_tombs, d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, stream));
  KVB_CUDA_TRY(cudaStreamSynchronize(stream));
  zero_tombs.tombs = 0;
  KVB_CUDA_TRY(cudaMemcpy(d_ctr, &zero_tombs, sizeof(Counters), cudaMemcpyHostToDevice));
  cudaFree(table);
  cudaFree(ts);
  table = fresh;
  ts = fresh_ts;
  slots = new_slots;
  h_ctr = zero_tombs;
  live_ub = (int64_t)h_ctr.live + q_adds;
  tomb_ub = q_evicts;
  order_valid = false;  // slots moved
  ++n_rehash;
  return KVB_OK;
}

// (stamp, slot) of every live key sorted by stamp: the outer LRU order at this moment.  Later stamps only make
// records stale, and keys inserted later are newer than every valid record, so the array serves until it runs out.
int kvb_index::ensure_sort_tmp(size_t need) {
  if (need <= sort_tmp_bytes) return KVB_OK;
  if (d_sort_tmp) cudaFree(d_sort_tmp);
  d_sort_tmp = nullptr;
  sort_tmp_bytes = 0;
  KVB_CUDA_TRY(cudaMalloc(&d_sort_tmp, need));
  sort_tmp_bytes = need;
  return KVB_OK;
}

// `min_records`: how many evictions the coming batch can ask for — an array with fewer records left is rebuilt now
// (running out inside a batch costs a whole-table scan per eviction on the sequential path).
int kvb_index::ensure_order(int64_t min_records) {
  if (order_valid) {
    const int64_t left = order_n - (int64_t)h_ctr.order_head;
    if (left >= std::min<int64_t>(std::max<int64_t>(min_records, 1), (int64_t)h_ctr.live)) return KVB_OK;
  }
  int rc = sync_counters();
  if (rc) return rc;
  const int64_t live = (int64_t)h_ctr.live;
  if (live > order_cap) {
    for (void* p : {(void*)order_ts, (void*)order_slot, (void*)order_ts_in, (void*)order_slot_in})
      if (p) cudaFree(p);
    order_ts = order_ts_in = nullptr;
    order_slot = order_slot_in = nullptr;
    order_cap = 0;
    const int64_t cap = std::max<int64_t>(live * 5 / 4, 1024);
    KVB_CUDA_TRY(cudaMalloc(&order_ts, cap * sizeof(unsigned long long)));
    KVB_CUDA_TRY(cudaMalloc(&order_ts_in, cap * sizeof(unsigned long long)));
    KVB_CUDA_TRY(cudaMalloc(&order_slot, cap * sizeof(uint32_t)));
    KVB_CUDA_TRY(cudaMalloc(&order_slot_in, cap * sizeof(uint32_t)));
    order_cap = cap;
  }
  if (!d_cursor) KVB_CUDA_TRY(cudaMalloc(&d_cursor, sizeof(unsigned long long)));
  KVB_CUDA_TRY(cudaMemsetAsync(d_cursor, 0, sizeof(unsigned long long), stream));
  const unsigned threads = 256;
  KVB_LAUNCH(index_collect_order_kernel, (unsigned)((slots + threads - 1) / threads), threads, stream, ref(),
             order_ts_in, order_slot_in, d_cursor, (unsigned long long)order_cap);
  KVB_CUDA_TRY(cudaGetLastError());
  count_launch();
  order_n = live;
  if (live > 0) {
#ifdef KVB_HOST_SIM
    sim_sort_pairs(order_ts_in, order_ts, order_slot_in, order_slot, live);
#else
    size_t need = 0;
    KVB_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, order_ts_in, order_ts, order_slot_in, order_slot,
                                                 (int)live, 0, 64, stream));
    rc = ensure_sort_tmp(need);
    if (rc) return rc;
    need = sort_tmp_bytes;
    KVB_CUDA_TRY(cub::DeviceRadixSort::SortPairs(d_sort_tmp, need, order_ts_in, order_ts, order_slot_in, order_slot,
                                                 (int)live, 0, 64, stream));
    count_launch();
#endif
  }
  Counters c = h_ctr;
  c.order_head = 0;
  KVB_CUDA_TRY(cudaStreamSynchronize(stream));
  KVB_CUDA_TRY(cudaMemcpy(d_ctr, &c, sizeof(Counters), cudaMemcpyHostToDevice));
  h_ctr = c;
  order_valid = true;
  ++n_order_builds;
  return KVB_OK;
}

// Victims of a batch at capacity, planned before anything is applied (see index_plan_events_kernel).
// *ok = false: the batch needs the one-thread replay (the order array cannot supply enough records even after a
// rebuild — an index smaller than the batch — or the plan did not settle).
int kvb_index::plan_evictions(int64_t n, int64_t* n_victims, unsigned long long* new_head, unsigned long long* skipped,
                              bool* ok) {
  *ok = false;
  *n_victims = 0;
  if (!d_plan_ops) KVB_CUDA_TRY(cudaMalloc(&d_plan_ops, 4 * kOpsCap * sizeof(uint32_t)));  // ev | net | top | evict_op
  if (!d_victims) KVB_CUDA_TRY(cudaMalloc(&d_victims, kOpsCap * sizeof(uint32_t)));
  if (!d_win) KVB_CUDA_TRY(cudaMalloc(&d_win, 3 * kWinCap * sizeof(uint32_t)));
  if (!d_plan) KVB_CUDA_TRY(cudaMalloc(&d_plan, 8 * sizeof(unsigned long long)));
  if (!d_conflict) KVB_CUDA_TRY(cudaMalloc(&d_conflict, 2 * kOpsCap));
  const unsigned threads = 128;
  const unsigned grid_n = (unsigned)((n + threads - 1) / threads);
  int32_t* ev = reinterpret_cast<int32_t*>(d_plan_ops);
  int32_t* net = ev + kOpsCap;
  int32_t* top = net + kOpsCap;
  uint32_t* evict_op = d_plan_ops + 3 * kOpsCap;
  uint32_t *is_victim = d_win, *touch = d_win + kWinCap, *rank = d_win + 2 * kWinCap;
  uint8_t *conf_cur = d_conflict, *conf_next = d_conflict + kOpsCap;
  KVB_CUDA_TRY(cudaMemsetAsync(conf_cur, 0, (size_t)n, stream));
  const int64_t live0 = (int64_t)h_ctr.live;  // exact: read after the last launch that changes it
  if (live0 > max_keys) return KVB_OK;
  unsigned long long h_plan[4] = {};
  int64_t n_conflicts = 0;
  bool rebuilt = false;
  static const bool plan_debug = getenv("KVB_PLAN_DEBUG") != nullptr;
  for (int iter = 0; iter < 24; ++iter) {
    // which ops insert / delete a key under the current conflict set, and from that the op of every eviction
    KVB_CUDA_TRY(cudaMemsetAsync(ev, 0, (size_t)n * sizeof(int32_t), stream));
    KVB_LAUNCH(index_plan_events_kernel, grid_n, threads, stream, ref(), d_ops, d_ents, d_skey_out, d_sidx_out, n,
               conf_cur, ev);
    KVB_CUDA_TRY(cudaGetLastError());
    int32_t top_last = 0;
#ifdef KVB_HOST_SIM
    for (int64_t i = 0, acc = 0, mx = INT32_MIN; i < n; ++i) {
      acc += ev[i];
      mx = std::max<int64_t>(mx, acc);
      net[i] = (int32_t)acc;
      top[i] = (int32_t)mx;
    }
    top_last = top[n - 1];
#else
    {
      size_t need = 0, need2 = 0;
      KVB_CUDA_TRY(cub::DeviceScan::InclusiveSum(nullptr, need, ev, net, (int)n, stream));
      KVB_CUDA_TRY(cub::DeviceScan::InclusiveScan(nullptr, need2, net, top, cub::Max(), (int)n, stream));
      int rc = ensure_sort_tmp(std::max(need, need2));
      if (rc) return rc;
      need = need2 = sort_tmp_bytes;
      KVB_CUDA_TRY(cub::DeviceScan::InclusiveSum(d_sort_tmp, need, ev, net, (int)n, stream));
      KVB_CUDA_TRY(cub::DeviceScan::InclusiveScan(d_sort_tmp, need2, net, top, cub::Max(), (int)n, stream));
      KVB_CUDA_TRY(cudaMemcpyAsync(&top_last, top + (n - 1), sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
      KVB_CUDA_TRY(cudaStreamSynchronize(stream));
    }
#endif
    count_launch(3);
    const int64_t want = std::max<int64_t>(0, live0 + std::max<int64_t>(top_last, 0) - max_keys);
    if (want == 0) {  // live never passes Size under this conflict set (which is then empty: nothing was evicted)
      if (n_conflicts != 0) return KVB_OK;
      *ok = true;
      *new_head = h_ctr.order_head;
      *skipped = 0;
      return KVB_OK;
    }
    KVB_LAUNCH(index_evict_times_kernel, grid_n, threads, stream, ev, net, top, n, live0, (int64_t)max_keys, evict_op);
    KVB_CUDA_TRY(cudaGetLastError());
    KVB_CUDA_TRY(cudaMemsetAsync(conf_next, 0, (size_t)n, stream));
    KVB_CUDA_TRY(cudaMemsetAsync(d_plan + 3, 0, sizeof(unsigned long long), stream));
    const int64_t head0 = (int64_t)h_ctr.order_head;
    int64_t pos = head0, found = 0, end = -1, changed = 0;
    while (found < want && pos < order_n) {
      const int64_t w = std::min<int64_t>(order_n - pos, std::min<int64_t>(kWinCap, std::max<int64_t>(2 * (want - found), 65536)));
      const unsigned grid = (unsigned)((w + threads - 1) / threads);
      KVB_CUDA_TRY(cudaMemsetAsync(d_plan, 0, 3 * sizeof(unsigned long long), stream));
      KVB_LAUNCH(index_evict_flag_kernel, grid, threads, stream, ref(), order_ts, order_slot, pos, w, d_skey_out, n,
                 conf_cur, is_victim, touch);
      KVB_CUDA_TRY(cudaGetLastError());
#ifdef KVB_HOST_SIM
      for (int64_t p = 0, acc = 0; p < w; ++p) {
        rank[p] = (uint32_t)acc;
        acc += is_victim[p];
      }
#else
      size_t need = 0;
      KVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, is_victim, rank, (int)w, stream));
      int rc = ensure_sort_tmp(need);
      if (rc) return rc;
      need = sort_tmp_bytes;
      KVB_CUDA_TRY(cub::DeviceScan::ExclusiveSum(d_sort_tmp, need, is_victim, rank, (int)w, stream));
#endif
      KVB_LAUNCH(index_evict_decide_kernel, grid, threads, stream, is_victim, touch, rank, w, pos, order_slot,
                 d_sidx_out, found, want - found, evict_op, conf_next, d_victims, d_plan);
      KVB_CUDA_TRY(cudaGetLastError());
      count_launch(3);
      KVB_CUDA_TRY(cudaMemcpyAsync(h_plan, d_plan, sizeof(h_plan), cudaMemcpyDeviceToHost, stream));
      KVB_CUDA_TRY(cudaStreamSynchronize(stream));
      changed += (int64_t)h_plan[0];
      found += (int64_t)h_plan[2];
      if (found >= want) {
        end = pos + (int64_t)h_plan[1];
        break;
      }
      pos += w;
    }
    const int64_t next_conflicts = (int64_t)h_plan[3];
    if (plan_debug)
      fprintf(stderr, "plan n %lld live %lld iter %d: want %lld found %lld end %lld changed %lld conflicts %lld -> %lld head %lld order_n %lld\n",
              (long long)n, (long long)live0, iter, (long long)want, (long long)found, (long long)end, (long long)changed,
              (long long)n_conflicts, (long long)next_conflicts, (long long)head0, (long long)order_n);
    if (end >= 0 && changed == 0 && next_conflicts == n_conflicts) {  // the plan reproduces itself: these are the victims
      *ok = true;
      *n_victims = want;
      *new_head = (unsigned long long)end;
      *skipped = (unsigned long long)(end - head0 - want);
      return KVB_OK;
    }
    if (end < 0 && changed == 0 && next_conflicts == n_conflicts) {
      // a settled plan that ran out of records: stale ones (lookups re-stamp keys) may have used the array up
      if (rebuilt) return KVB_OK;
      rebuilt = true;
      order_valid = false;
      int rc = ensure_order();
      if (rc) return rc;
      continue;
    }
    std::swap(conf_cur, conf_next);
    n_conflicts = next_conflicts;
  }
  return KVB_OK;
}

int kvb_index::flush_locked() {
  if (n_ops == 0) return KVB_OK;
  // grow before the table gets crowded: live + tombstones + incoming <= 0.6 * slots (bounds first, exact if they trip)
  if ((uint64_t)(live_ub + tomb_ub) * 10 > slots * 6) {
    int rc = sync_counters();
    if (rc) return rc;
    if ((uint64_t)(live_ub + tomb_ub) * 10 > slots * 6) {
      uint64_t ns = slots;
      while ((uint64_t)live_ub * 10 > ns * 3) ns <<= 1;  // target load <= 0.3 after the move
      rc = rehash(ns);                                   // same size: only drops the tombstones
      if (rc) return rc;
    }
  }
  bool may_evict = live_ub > max_keys;
  if (may_evict) {
    int rc = sync_counters();
    if (rc) return rc;
    may_evict = live_ub > max_keys;
  }
  KVB_CUDA_TRY(cudaMemcpyAsync(d_ents, h_ents, n_ents * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
  // At capacity a queue longer than half the index is applied in pieces of that length, each a batch of its own: a piece
  // never needs more victims than the freshly built order array holds untouched records (Size - piece >= piece), so the
  // eviction plan always has what it needs and the one-thread replay never has to scan the table for a minimum —
  // except for indexes of a handful of keys, where the scan is a handful of slots.
  size_t piece = n_ops;
  if (may_evict && (int64_t)n_ops > max_keys / 2) piece = (size_t)std::max<int64_t>(max_keys / 2, 1);
  for (size_t first = 0; first < n_ops; first += piece) {
    int rc = flush_piece(first, std::min(piece, n_ops - first), may_evict);
    if (rc) return rc;
  }
  KVB_CUDA_TRY(cudaEventRecord(q_free, stream));
  q_busy = true;
  n_ops_total += (int64_t)n_ops;
  n_ops = n_ents = 0;
  q_adds = q_evicts = 0;  // they stay counted inside live_ub / tomb_ub until the next exact read
  if (may_evict) {
    int rc = sync_counters();  // the order head moved; exact counts keep the bounds from drifting at capacity
    if (rc) return rc;
  }
  return KVB_OK;
}

// ops [first, first + count) of the pinned queue as one batch
int kvb_index::flush_piece(size_t first, size_t count, bool may_evict) {
  const bool small = (int64_t)count <= kSeqThreshold;
  // at capacity a batch still runs in parallel, with its evictions planned up front (plan_evictions); the one-thread
  // replay in the reference's order remains for tiny batches and for plans that do not settle
  static const bool plan_off = getenv("KVB_INDEX_PLAN") != nullptr && getenv("KVB_INDEX_PLAN")[0] == '0';
  bool planned = may_evict && !small && !plan_off;
  bool sequential = small || (may_evict && !planned);
  if (may_evict) {
    int rc = first ? sync_counters() : KVB_OK;  // the previous piece moved the counters and the order head
    if (rc == KVB_OK) rc = ensure_order((int64_t)count);
    if (rc) return rc;
  }
  KVB_CUDA_TRY(cudaMemcpyAsync(d_ops, h_ops + first, count * sizeof(OpRec), cudaMemcpyHostToDevice, stream));
  const unsigned long long seq_base = seq;
  seq += count;
  const int64_t n = (int64_t)count;
  const unsigned threads = 128;
  const unsigned grid = (unsigned)((n + threads - 1) / threads);
  int64_t n_victims = 0;
  unsigned long long new_head = 0, skipped = 0;
  if (!sequential) {
    KVB_LAUNCH(index_sort_keys_kernel, grid, threads, stream, d_ops, n, d_skey_in, d_sidx_in);
    KVB_CUDA_TRY(cudaGetLastError());
#ifdef KVB_HOST_SIM
    sim_sort_pairs(d_skey_in, d_skey_out, d_sidx_in, d_sidx_out, n);
#else
    size_t need = sort_tmp_bytes;
    cudaError_t e = cub::DeviceRadixSort::SortPairs(d_sort_tmp, need, d_skey_in, d_skey_out, d_sidx_in, d_sidx_out,
                                                    (int)n, 0, 64, stream);
    if (e != cudaSuccess) {
      set_error("index: sorting %lld ops failed: %s", (long long)n, cudaGetErrorString(e));
      return KVB_ERR_CUDA;
    }
#endif
    count_launch(2);
    if (planned) {
      bool ok = false;
      int rc = plan_evictions(n, &n_victims, &new_head, &skipped, &ok);
      if (rc) return rc;
      if (!ok) {
        sequential = true;
        planned = false;
        ++n_plan_fallbacks;
      }
    }
  }
  if (sequential) {
    // a table of up to this many slots may be scanned for its oldest key when the order array runs out inside the
    // replay; above it the replay stops, the order array is rebuilt and the replay resumes
    static const unsigned long long scan_max_slots =
        getenv("KVB_INDEX_SCAN_MAX_SLOTS") ? strtoull(getenv("KVB_INDEX_SCAN_MAX_SLOTS"), nullptr, 10) : 65536ull;
    for (int64_t start = 0; start >= 0;) {
      KVB_LAUNCH(index_apply_seq_kernel, 1, 1, stream, ref(), d_ops, d_ents, start, n, seq_base,
                 (unsigned long long)max_keys, order_ts, order_slot, (unsigned long long)(may_evict ? order_n : 0),
                 scan_max_slots);
      KVB_CUDA_TRY(cudaGetLastError());
      count_launch();
      start = -1;
      if (may_evict && slots > scan_max_slots) {
        int rc = sync_counters();
        if (rc) return rc;
        if (h_ctr.resume_at >= 0 || h_ctr.pending_evict) {
          start = h_ctr.resume_at >= 0 ? h_ctr.resume_at : n;
          order_valid = false;
          rc = ensure_order();
          if (rc) return rc;
          ++n_seq_resumes;
        }
      }
    }
    ++n_flush_seq;
  } else {
    if (planned) {  // victims go first: a conflict key must be absent when its ops are replayed
      ++n_flush_planned;
      if (n_victims > 0) {
        KVB_LAUNCH(index_evict_apply_kernel, (unsigned)((n_victims + threads - 1) / threads), threads, stream, ref(),
                   d_victims, n_victims, new_head, skipped);
        KVB_CUDA_TRY(cudaGetLastError());
        count_launch();
      }
    }
    KVB_LAUNCH(index_apply_par_kernel, grid, threads, stream, ref(), d_ops, d_ents, d_skey_out, d_sidx_out, n,
               seq_base);
    KVB_CUDA_TRY(cudaGetLastError());
    count_launch();
    ++n_flush_par;
  }
  return KVB_OK;
}

int kvb_index::queue_ops(uint8_t type, const uint64_t* keys, int64_t n_keys, const kvb_pod_entry_t* entries,
                         int32_t n_entries) {
  int64_t done = 0;
  while (done < n_keys) {
    if (n_ops == kOpsCap || n_ents + (size_t)n_entries > kEntsCap) {
      int rc = flush_locked();
      if (rc) return rc;
    }
    if (q_busy) {  // the pinned queue is still being read by the previous flush's copies
      KVB_CUDA_TRY(cudaEventSynchronize(q_free));
      q_busy = false;
    }
    const uint32_t ent_off = (uint32_t)n_ents;
    for (int32_t e = 0; e < n_entries; ++e)
      h_ents[n_ents++] = pack_entry(entries[e].pod, entries[e].tier, entries[e].speculative);
    const int64_t take = std::min<int64_t>(n_keys - done, (int64_t)(kOpsCap - n_ops));
    for (int64_t i = 0; i < take; ++i) {
      OpRec& r = h_ops[n_ops++];
      r.key = keys[done + i];
      r.ent_off = ent_off;
      r.ent_cnt = (uint16_t)n_entries;
      r.type = type;
      r.pad = 0;
    }
    if (type == kOpAdd) {
      q_adds += take;
      live_ub += take;
    } else {
      q_evicts += take;
      tomb_ub += take;
    }
    done += take;
  }
  return KVB_OK;
}

// pod filter bitmap (65536 bits), resident on the device and re-uploaded only when the filter changes.  When it does
// change the bitmap is written into the caller's pinned staging block (*staged = true) and copied from there on the
// stream — no synchronisation, the staging block outlives the call's own stream sync.
int kvb_index::set_filter(const uint16_t* pods, int32_t n, uint8_t* h_stage, bool* staged, const uint32_t** out) {
  *out = nullptr;
  *staged = false;
  if (n <= 0) return KVB_OK;
  if (!d_filter) KVB_CUDA_TRY(cudaMalloc(&d_filter, 2048 * sizeof(uint32_t)));
  *out = d_filter;
  if (filter_valid && filter_cached.size() == (size_t)n && std::memcmp(filter_cached.data(), pods, (size_t)n * 2) == 0)
    return KVB_OK;
  uint32_t* bits = reinterpret_cast<uint32_t*>(h_stage);
  std::memset(bits, 0, 2048 * sizeof(uint32_t));
  for (int32_t i = 0; i < n; ++i) bits[pods[i] >> 5] |= 1u << (pods[i] & 31);
  KVB_CUDA_TRY(cudaMemcpyAsync(d_filter, bits, 2048 * sizeof(uint32_t), cudaMemcpyHostToDevice, stream));
  filter_cached.assign(pods, pods + n);
  filter_valid = true;
  *staged = true;
  return KVB_OK;
}

// kvb_index_remove_pods under the lock: queued ops first, then one sweep of the table.  Deleting keys turns live slots
// into tombstones (live + tombs stays put), so no rehash is due here; flush_locked's growth rule stays the only one.
int kvb_index::remove_pods_locked(const uint16_t* pods, int32_t n_pods, const uint8_t* tiers, int32_t n_tiers,
                                  int64_t* entries_removed, int64_t* keys_deleted) {
  int rc = flush_locked();
  if (rc) return rc;
  constexpr size_t kBitsBytes = 2048 * sizeof(uint32_t);
  rc = ensure_scratch(0, kBitsBytes);
  if (rc) return rc;
  if (!d_purge_bits) KVB_CUDA_TRY(cudaMalloc(&d_purge_bits, kBitsBytes));
  uint32_t* bits = reinterpret_cast<uint32_t*>(h_scratch);
  std::memset(bits, 0, kBitsBytes);
  for (int32_t i = 0; i < n_pods; ++i) bits[pods[i] >> 5] |= 1u << (pods[i] & 31);
  TierMask tm;
  std::memset(&tm, n_tiers > 0 ? 0 : 0xff, sizeof(tm));
  for (int32_t i = 0; i < n_tiers; ++i) tm.bits[tiers[i] >> 5] |= 1u << (tiers[i] & 31);
  KVB_CUDA_TRY(cudaMemcpyAsync(d_purge_bits, bits, kBitsBytes, cudaMemcpyHostToDevice, stream));
  KVB_CUDA_TRY(cudaMemsetAsync(&d_ctr->purge_entries, 0, 2 * sizeof(unsigned long long), stream));
  const uint64_t per_block = (uint64_t)kPurgeThreads * kPurgeUnroll;
  uint64_t grid = (slots + per_block - 1) / per_block;
#ifndef KVB_HOST_SIM
  static int blocks_per_sm = 0;
  if (blocks_per_sm == 0)
    KVB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocks_per_sm, index_remove_pods_kernel, kPurgeThreads, 0));
  grid = std::min<uint64_t>(grid, (uint64_t)sm_count(device) * (uint64_t)std::max(blocks_per_sm, 1));
#endif
  KVB_LAUNCH(index_remove_pods_kernel, (unsigned)grid, kPurgeThreads, stream, ref(), d_purge_bits, tm);
  KVB_CUDA_TRY(cudaGetLastError());
  count_launch();
  rc = sync_counters();  // live_ub / tomb_ub exact again
  if (rc) return rc;
  // the LRU order array is rebuilt the next time the index is at capacity; its records of freed slots are stale anyway
  if (h_ctr.purge_keys) order_valid = false;
  if (entries_removed) *entries_removed = (int64_t)h_ctr.purge_entries;
  if (keys_deleted) *keys_deleted = (int64_t)h_ctr.purge_keys;
  return KVB_OK;
}

// engineKey -> requestKeys mapping of one Add (in_memory.go:166-177): ek = engine[i*|E|/n], rk = request[i*|R|/n], n = max
static void map_engine_keys(EngMap& em, const uint64_t* engine_keys, int64_t n_engine, const uint64_t* request_keys,
                            int64_t n_request) {
  bool one_to_one = n_engine == n_request;  // the common shape: one request key per engine key, no repeats
  if (one_to_one && n_engine > 1) {
    std::vector<uint64_t> sorted(engine_keys, engine_keys + n_engine);
    std::sort(sorted.begin(), sorted.end());
    one_to_one = std::adjacent_find(sorted.begin(), sorted.end()) == sorted.end();
  }
  if (one_to_one) {
    for (int64_t i = 0; i < n_engine; ++i) em.put(engine_keys[i], &request_keys[i], 1);
    return;
  }
  const int64_t n = std::max(n_engine, n_request);
  std::vector<uint64_t> order;
  std::unordered_map<uint64_t, std::vector<uint64_t>> m;
  for (int64_t i = 0; i < n; ++i) {
    const uint64_t ek = engine_keys[i * n_engine / n];
    const uint64_t rk = request_keys[i * n_request / n];
    auto it = m.find(ek);
    if (it == m.end()) {
      order.push_back(ek);
      m[ek].push_back(rk);
    } else {
      it->second.push_back(rk);
    }
  }
  // Go iterates newMappings in random order (in_memory.go:174-176); first-seen order here (only observable when the
  // engine-key LRU is at capacity)
  for (uint64_t ek : order) {
    const auto& v = m[ek];
    em.put(ek, v.data(), v.size());
  }
}

extern "C" {

int kvb_index_create(int device, int64_t max_keys, int32_t pods_per_key, int64_t expected_keys, kvb_index_t** out) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(out != nullptr, "out is NULL");
    *out = nullptr;
    KVB_REQUIRE(max_keys > 0, "must provide a positive size");  // golang-lru New()
    KVB_REQUIRE(pods_per_key > 0, "must provide a positive size");
    if (pods_per_key > kMaxEnt) {
      set_error("podCacheSize %d exceeds the %d entries of a device bucket", pods_per_key, kMaxEnt);
      return KVB_ERR_UNSUPPORTED;
    }
    DeviceGuard g(device);
    if (!g.ok) {
      set_error("cannot select CUDA device %d", device);
      return KVB_ERR_CUDA;
    }
    // kvb_index_destroy releases whatever CUDA resources exist if a later step fails
    std::unique_ptr<kvb_index, void (*)(kvb_index*)> idx(new kvb_index(), kvb_index_destroy);
    idx->device = device;
    idx->max_keys = max_keys;
    idx->pods_per_key = pods_per_key;
    idx->eng.reset(new EngMap(max_keys));
    for (int i = 0; i < 256; ++i) idx->tier_w_host[i] = 1.0;  // unknown tier -> 1.0 (kvblock_scorer.go:93-98)
    KVB_CUDA_TRY(cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking));
    KVB_CUDA_TRY(cudaEventCreateWithFlags(&idx->q_free, cudaEventDisableTiming));
    KVB_CUDA_TRY(cudaEventCreateWithFlags(&idx->ev_a, cudaEventDefault));
    KVB_CUDA_TRY(cudaEventCreateWithFlags(&idx->ev_b, cudaEventDefault));
    KVB_CUDA_TRY(cudaEventCreateWithFlags(&idx->ev_c, cudaEventDefault));
#ifndef KVB_HOST_SIM
    idx->spec = spec_scratch_create();
#endif
    KVB_CUDA_TRY(cudaMalloc(&idx->tier_w, 256 * sizeof(double)));
    KVB_CUDA_TRY(cudaMemcpy(idx->tier_w, idx->tier_w_host, 256 * sizeof(double), cudaMemcpyHostToDevice));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_ctr, sizeof(Counters)));
    KVB_CUDA_TRY(cudaMemset(idx->d_ctr, 0, sizeof(Counters)));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_done, sizeof(unsigned)));
    KVB_CUDA_TRY(cudaMemset(idx->d_done, 0, sizeof(unsigned)));
    KVB_CUDA_TRY(host_alloc_near(device, reinterpret_cast<void**>(&idx->h_done), 64, cudaHostAllocPortable | cudaHostAllocMapped));
    *idx->h_done = 0ull;
    int64_t exp_keys = std::max<int64_t>(expected_keys, 1024);
    exp_keys = std::min<int64_t>(exp_keys, max_keys);
    uint64_t slots = 2048;
    while (slots * 3 < (uint64_t)exp_keys * 10) slots <<= 1;  // load <= 0.3 at expected size
    idx->slots = slots;
    int rc = idx->alloc_table(slots, &idx->table, &idx->ts);
    if (rc) return rc;
    // op queue: pinned on the GPU's NUMA node; device copies and sort buffers sized for a full queue
    KVB_CUDA_TRY(host_alloc_near(device, reinterpret_cast<void**>(&idx->h_ops), kvb_index::kOpsCap * sizeof(OpRec),
                                 cudaHostAllocPortable));
    KVB_CUDA_TRY(host_alloc_near(device, reinterpret_cast<void**>(&idx->h_ents), kvb_index::kEntsCap * sizeof(uint32_t),
                                 cudaHostAllocPortable));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_ops, kvb_index::kOpsCap * sizeof(OpRec)));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_ents, kvb_index::kEntsCap * sizeof(uint32_t)));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_skey_in, kvb_index::kOpsCap * sizeof(uint64_t)));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_skey_out, kvb_index::kOpsCap * sizeof(uint64_t)));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_sidx_in, kvb_index::kOpsCap * sizeof(uint32_t)));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_sidx_out, kvb_index::kOpsCap * sizeof(uint32_t)));
#ifndef KVB_HOST_SIM
    size_t need = 0;
    KVB_CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, idx->d_skey_in, idx->d_skey_out, idx->d_sidx_in,
                                                 idx->d_sidx_out, (int)kvb_index::kOpsCap, 0, 64, idx->stream));
    KVB_CUDA_TRY(cudaMalloc(&idx->d_sort_tmp, need));
    idx->sort_tmp_bytes = need;
#endif
    KVB_CUDA_TRY(cudaStreamSynchronize(idx->stream));
    *out = idx.release();
    return KVB_OK;
  });
}

void kvb_index_destroy(kvb_index_t* idx) {
  if (!idx) return;
  DeviceGuard g(idx->device);
  if (idx->stream) cudaStreamSynchronize(idx->stream);
  for (void* p : {(void*)idx->table, (void*)idx->ts, (void*)idx->d_ctr, (void*)idx->tier_w, (void*)idx->d_ops,
                  (void*)idx->d_ents, (void*)idx->d_skey_in, (void*)idx->d_skey_out, (void*)idx->d_sidx_in,
                  (void*)idx->d_sidx_out, idx->d_sort_tmp, (void*)idx->order_ts, (void*)idx->order_slot,
                  (void*)idx->order_ts_in, (void*)idx->order_slot_in, (void*)idx->d_cursor, (void*)idx->d_scratch,
                  (void*)idx->d_filter, (void*)idx->d_done, (void*)idx->d_plan_ops, (void*)idx->d_victims,
                  (void*)idx->d_win, (void*)idx->d_plan, (void*)idx->d_conflict, (void*)idx->d_purge_bits})
    if (p) cudaFree(p);
  for (void* p : {(void*)idx->h_ops, (void*)idx->h_ents, (void*)idx->h_scratch, (void*)idx->h_done})
    if (p) cudaFreeHost(p);
  for (cudaEvent_t e : {idx->q_free, idx->ev_a, idx->ev_b, idx->ev_c})
    if (e) cudaEventDestroy(e);
#ifndef KVB_HOST_SIM
  spec_scratch_destroy(idx->spec);
#endif
  if (idx->stream) cudaStreamDestroy(idx->stream);
  delete idx;
}

int kvb_index_set_tier_weight(kvb_index_t* idx, uint8_t tier, double weight, int known) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    idx->tier_w_host[tier] = known ? weight : 1.0;
    KVB_CUDA_TRY(cudaStreamSynchronize(idx->stream));  // no scoring kernel may be reading the table
    KVB_CUDA_TRY(cudaMemcpy(idx->tier_w + tier, &idx->tier_w_host[tier], sizeof(double), cudaMemcpyHostToDevice));
    return KVB_OK;
  });
}

int kvb_index_add(kvb_index_t* idx, const uint64_t* engine_keys, int64_t n_engine, int has_engine_keys,
                  const uint64_t* request_keys, int64_t n_request, const kvb_pod_entry_t* entries, int32_t n_entries) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    // in_memory.go:155-157
    KVB_REQUIRE(n_request > 0 && n_entries > 0 && request_keys && entries,
                "no keys or entries provided for adding to index");
    KVB_REQUIRE(!has_engine_keys || n_engine > 0, "engineKeys is non-nil but empty");
    KVB_REQUIRE(n_entries <= 65535, "too many entries in one Add");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    if (has_engine_keys) map_engine_keys(*idx->eng, engine_keys, n_engine, request_keys, n_request);  // in_memory.go:166-177
    return idx->queue_ops(kOpAdd, request_keys, n_request, entries, n_entries);  // in_memory.go:180-221
  });
}

int kvb_index_evict(kvb_index_t* idx, uint64_t key, int key_type, const kvb_pod_entry_t* entries, int32_t n_entries) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    KVB_REQUIRE(n_entries > 0 && entries, "no entries provided for eviction from index");  // in_memory.go:230-232
    KVB_REQUIRE(n_entries <= 65535, "too many entries in one Evict");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    if (key_type == KVB_KEY_ENGINE) {
      EngMap& em = *idx->eng;
      const int64_t id = em.find(key);
      if (id < 0) return KVB_OK;  // nothing to evict (in_memory.go:238-242)
      std::vector<uint64_t> rks;
      em.for_each_rk(id, [&](uint64_t rk) { rks.push_back(rk); });
      em.erase(id);  // in_memory.go:247
      if (rks.empty()) return KVB_OK;
      return idx->queue_ops(kOpEvict, rks.data(), (int64_t)rks.size(), entries, n_entries);
    }
    if (key_type == KVB_KEY_REQUEST) return idx->queue_ops(kOpEvict, &key, 1, entries, n_entries);
    set_error("unknown key type: %d", key_type);  // in_memory.go:252-254
    return KVB_ERR_INVALID;
  });
}

int kvb_index_remove_pods(kvb_index_t* idx, const uint16_t* pods, int32_t n_pods, const uint8_t* tiers, int32_t n_tiers,
                          int64_t* out_entries_removed, int64_t* out_keys_deleted) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    KVB_REQUIRE(n_pods >= 1 && pods, "no pods provided for removal from index");
    KVB_REQUIRE(n_tiers >= 0 && (n_tiers == 0 || tiers), "bad tier list");
    if (!tiers) n_tiers = 0;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    return idx->remove_pods_locked(pods, n_pods, tiers, n_tiers, out_entries_removed, out_keys_deleted);
  });
}

int kvb_index_get_request_key(kvb_index_t* idx, uint64_t engine_key, uint64_t* out) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx && out, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    const int64_t id = idx->eng->find(engine_key);
    if (id < 0 || idx->eng->node(id).n == 0) {  // in_memory.go:299-302
      set_error("engine key not found: %llu", (unsigned long long)engine_key);
      *out = 0;
      return KVB_ERR_NOTFOUND;
    }
    idx->eng->touch(id);
    *out = idx->eng->node(id).rk_last;
    return KVB_OK;
  });
}

#ifndef KVB_HOST_SIM
// Pool.processEventBatch (pkg/kvevents/pool.go:253-398) for a decoded batch, inside the library: per round, the next event of
// every stream (= pod; a pod's events stay in order, pods are independent — the reference runs them on parallel worker shards,
// pool.go:154-166).  BlockRemoved events evict through the engine-key map; the round's BlockStored events resolve their parents
// (GetRequestKey, pool.go:284-294), are hashed in ONE device launch, and are added (engine map on the host, bucket ops queued
// for the device).  Nothing returns to the host language per event.
int kvb_index_ingest_events(kvb_index_t* idx, const kvb_kv_event_t* ev, int32_t n_events, const uint32_t* tokens,
                            const uint64_t* engine_keys, int32_t block_size, int32_t* out_skipped) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    KVB_REQUIRE(n_events >= 0 && (n_events == 0 || ev), "bad event list");
    KVB_REQUIRE(block_size > 0, "blockSize must be greater than 0, got %d", block_size);
    if (out_skipped) *out_skipped = 0;
    if (n_events == 0) return KVB_OK;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    int32_t skipped = 0;
    // rounds: position of each event inside its stream
    std::unordered_map<int32_t, int32_t> seen;
    std::vector<std::vector<int32_t>> rounds;
    for (int32_t e = 0; e < n_events; ++e) {
      KVB_REQUIRE(ev[e].n_tokens >= 0 && ev[e].n_engine_keys >= 0, "event %d has negative sizes", e);
      const int32_t r = seen[ev[e].stream]++;
      if ((size_t)r >= rounds.size()) rounds.resize((size_t)r + 1);
      rounds[(size_t)r].push_back(e);
    }
    auto al = [](size_t x) { return (x + 255) & ~size_t(255); };
    std::vector<int32_t> stored;
    std::vector<uint64_t> keys_tmp;
    for (const auto& round : rounds) {
      stored.clear();
      int64_t tot_tok = 0, tot_keys = 0;
      for (int32_t e : round) {
        const kvb_kv_event_t& x = ev[e];
        if (x.type == KVB_EVENT_BLOCK_REMOVED) {  // pool.go:379-386: every engine key, ENGINE key type
          for (int64_t k = 0; k < x.n_engine_keys; ++k) {
            const int64_t id = idx->eng->find(engine_keys[x.engine_key_off + k]);
            if (id < 0) continue;
            keys_tmp.clear();
            idx->eng->for_each_rk(id, [&](uint64_t rk) { keys_tmp.push_back(rk); });
            idx->eng->erase(id);
            if (!keys_tmp.empty()) {
              int rc = idx->queue_ops(kOpEvict, keys_tmp.data(), (int64_t)keys_tmp.size(), &x.entry, 1);
              if (rc) return rc;
            }
          }
          continue;
        }
        if (x.type == KVB_EVENT_POD_CLEARED) {  // opt-in AllBlocksCleared: ops queued so far first, then the sweep
          int rc = idx->remove_pods_locked(&x.entry.pod, 1, &x.entry.tier, 1, nullptr, nullptr);
          if (rc) return rc;
          continue;
        }
        if (x.type != KVB_EVENT_BLOCK_STORED) continue;  // AllBlocksCleared and unknown events: log only (pool.go:388-395)
        if (x.n_tokens / block_size == 0 || x.n_engine_keys == 0) {
          ++skipped;  // "no request keys produced, skipping" (pool.go:350-355)
          continue;
        }
        stored.push_back(e);
        tot_tok += x.n_tokens;
        tot_keys += x.n_tokens / block_size;
      }
      if (stored.empty()) continue;
      const int32_t n = (int32_t)stored.size();
      // staging: [poff | koff | parents | tokens]  ->  device;  keys  <-  device
      size_t o = 0;
      const size_t o_poff = o;  o += al(((size_t)n + 1) * 8);
      const size_t o_koff = o;  o += al(((size_t)n + 1) * 8);
      const size_t o_par = o;   o += al((size_t)n * 8);
      const size_t o_tok = o;   o += al((size_t)tot_tok * 4);
      const size_t in_end = o;
      const size_t o_keys = o;  o += al((size_t)tot_keys * 8);
      int rc = idx->ensure_scratch(o, o);
      if (rc) return rc;
      uint8_t *H = idx->h_scratch, *D = idx->d_scratch;
      int64_t* h_poff = reinterpret_cast<int64_t*>(H + o_poff);
      int64_t* h_koff = reinterpret_cast<int64_t*>(H + o_koff);
      uint64_t* h_par = reinterpret_cast<uint64_t*>(H + o_par);
      uint32_t* h_tok = reinterpret_cast<uint32_t*>(H + o_tok);
      h_poff[0] = h_koff[0] = 0;
      int32_t m = 0;  // events that survive the parent lookup
      for (int32_t e : stored) {
        const kvb_kv_event_t& x = ev[e];
        uint64_t parent = x.root_hash;
        if (x.parent_engine_key != 0) {  // pool.go:284-294: unknown parent -> the event is dropped
          const int64_t id = idx->eng->find(x.parent_engine_key);
          if (id < 0 || idx->eng->node(id).n == 0) {
            ++skipped;
            continue;
          }
          idx->eng->touch(id);
          parent = idx->eng->node(id).rk_last;
        }
        h_par[m] = parent;
        std::memcpy(h_tok + h_poff[m], tokens + x.token_off, (size_t)x.n_tokens * 4);
        h_poff[m + 1] = h_poff[m] + x.n_tokens;
        h_koff[m + 1] = h_koff[m] + x.n_tokens / block_size;
        stored[(size_t)m] = e;
        ++m;
      }
      if (m == 0) continue;
      cudaStream_t s = idx->stream;
      KVB_CUDA_TRY(cudaMemcpyAsync(D, H, in_end, cudaMemcpyHostToDevice, s));
      rc = launch_hash_blocks(reinterpret_cast<uint32_t*>(D + o_tok), reinterpret_cast<int64_t*>(D + o_poff),
                              reinterpret_cast<uint64_t*>(D + o_par), m, block_size, nullptr, nullptr,
                              reinterpret_cast<uint64_t*>(D + o_keys), reinterpret_cast<int64_t*>(D + o_koff), s, h_koff[m], nullptr, nullptr, nullptr,
                              idx->spec);
      if (rc) return rc;
      KVB_CUDA_TRY(cudaMemcpyAsync(H + o_keys, D + o_keys, (size_t)h_koff[m] * 8, cudaMemcpyDeviceToHost, s));
      KVB_CUDA_TRY(cudaStreamSynchronize(s));
      const uint64_t* h_keys = reinterpret_cast<const uint64_t*>(H + o_keys);
      // the staging block is reused by the next round and by queue_ops' flushes: take the keys out first
      keys_tmp.assign(h_keys, h_keys + h_koff[m]);
      std::vector<int64_t> koff(h_koff, h_koff + m + 1);
      for (int32_t i = 0; i < m; ++i) {
        const kvb_kv_event_t& x = ev[stored[(size_t)i]];
        const uint64_t* rks = keys_tmp.data() + koff[(size_t)i];
        const int64_t n_rk = koff[(size_t)i + 1] - koff[(size_t)i];
        map_engine_keys(*idx->eng, engine_keys + x.engine_key_off, x.n_engine_keys, rks, n_rk);  // pool.go:360 Index.Add
        rc = idx->queue_ops(kOpAdd, rks, n_rk, &x.entry, 1);
        if (rc) return rc;
      }
    }
    if (out_skipped) *out_skipped = skipped;
    return KVB_OK;
  });
}
#endif  // !KVB_HOST_SIM

int64_t kvb_index_num_keys(kvb_index_t* idx) {
  if (!idx) return 0;
  int64_t n = 0;
  kvb::guarded([&]() -> int {
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    int rc = idx->flush_locked();
    if (rc == KVB_OK) rc = idx->sync_counters();
    n = rc == KVB_OK ? (int64_t)idx->h_ctr.live : 0;
    return rc;
  });
  return n;
}

int kvb_index_flush(kvb_index_t* idx, void* stream) {
  return kvb::guarded([&]() -> int {
    (void)stream;
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    int rc = idx->flush_locked();
    if (rc) return rc;
    KVB_CUDA_TRY(cudaStreamSynchronize(idx->stream));
    return KVB_OK;
  });
}

int kvb_index_get_stats(kvb_index_t* idx, kvb_index_stats_t* out) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx && out, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    int rc = idx->flush_locked();
    if (rc == KVB_OK) rc = idx->sync_counters();
    if (rc) return rc;
    std::memset(out, 0, sizeof(*out));
    out->live_keys = (int64_t)idx->h_ctr.live;
    out->tombstones = (int64_t)idx->h_ctr.tombs;
    out->table_slots = (int64_t)idx->slots;
    out->engine_keys = (int64_t)idx->eng->size();
    out->ops_applied = idx->n_ops_total;
    out->flushes_parallel = idx->n_flush_par;
    out->flushes_sequential = idx->n_flush_seq;
    out->flushes_planned = idx->n_flush_planned;
    out->plan_fallbacks = idx->n_plan_fallbacks;
    out->replay_resumes = idx->n_seq_resumes;
    out->rehashes = idx->n_rehash;
    out->lru_evictions = (int64_t)idx->h_ctr.evicted;
    out->order_builds = idx->n_order_builds;
    out->order_stale_skipped = (int64_t)idx->h_ctr.stale_skipped;
    out->order_scans = (int64_t)idx->h_ctr.scans;
    out->last_hash_us = idx->last_hash_us;
    out->last_score_us = idx->last_score_us;
    return KVB_OK;
  });
}

// shared by kvb_index_lookup and kvb_index_host_peek; caller holds the lock and the device
static int lookup_locked(kvb_index* idx, const uint64_t* keys, int64_t n, const uint16_t* pod_filter, int32_t n_filter,
                         bool stamp, const int32_t** cnt_out, const uint32_t** ent_out) {
  int rc = idx->flush_locked();
  if (rc) return rc;
  const size_t o_keys = 0, o_cnt = (size_t)n * 8, o_ent = o_cnt + (((size_t)n * 4 + 255) & ~size_t(255));
  const size_t o_filt = o_ent + (((size_t)n * kMaxEnt * 4 + 255) & ~size_t(255));
  const size_t total = o_filt + 2048 * sizeof(uint32_t);
  rc = idx->ensure_scratch(total, total);
  if (rc) return rc;
  const uint32_t* filt = nullptr;
  bool staged = false;
  rc = idx->set_filter(pod_filter, n_filter, idx->h_scratch + o_filt, &staged, &filt);
  if (rc) return rc;
  std::memcpy(idx->h_scratch, keys, (size_t)n * 8);
  cudaStream_t s = idx->stream;
  KVB_CUDA_TRY(cudaMemcpyAsync(idx->d_scratch + o_keys, idx->h_scratch, (size_t)n * 8, cudaMemcpyHostToDevice, s));
  unsigned long long stamp_base = 0ull;
  if (stamp) {
    stamp_base = idx->seq;
    idx->seq += (unsigned long long)n;
  }
  const int threads = 128;
  KVB_LAUNCH(index_lookup_kernel, (unsigned)((n + threads - 1) / threads), threads, s, idx->table, idx->slots - 1,
             reinterpret_cast<const uint64_t*>(idx->d_scratch + o_keys), n, filt,
             reinterpret_cast<int32_t*>(idx->d_scratch + o_cnt), reinterpret_cast<uint32_t*>(idx->d_scratch + o_ent),
             idx->ts, stamp_base);
  KVB_CUDA_TRY(cudaGetLastError());
  count_launch();
  KVB_CUDA_TRY(cudaMemcpyAsync(idx->h_scratch + o_cnt, idx->d_scratch + o_cnt, o_filt - o_cnt, cudaMemcpyDeviceToHost, s));
  KVB_CUDA_TRY(cudaStreamSynchronize(s));
  *cnt_out = reinterpret_cast<const int32_t*>(idx->h_scratch + o_cnt);
  *ent_out = reinterpret_cast<const uint32_t*>(idx->h_scratch + o_ent);
  return KVB_OK;
}

int kvb_index_host_peek(kvb_index_t* idx, uint64_t request_key, kvb_pod_entry_t* out_entries, int32_t cap) {
  int n_out = -1;
  kvb::guarded([&]() -> int {
    if (!idx) return KVB_OK;
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    const int32_t* cnt = nullptr;
    const uint32_t* ent = nullptr;
    int rc = lookup_locked(idx, &request_key, 1, nullptr, 0, false, &cnt, &ent);  // no recency refresh: a debug read
    if (rc) return rc;
    if (cnt[0] == -1) return KVB_OK;
    const int c = cnt[0] == -2 ? 0 : cnt[0];
    for (int i = 0; i < c && i < cap; ++i) {
      out_entries[i].pod = (uint16_t)(ent[i] & 0xffffu);
      out_entries[i].tier = (uint8_t)((ent[i] >> 16) & 0xffu);
      out_entries[i].speculative = (uint8_t)((ent[i] >> 24) & 1u);
    }
    n_out = c;
    return KVB_OK;
  });
  return n_out;
}

int kvb_index_lookup(kvb_index_t* idx, const uint64_t* keys, int64_t n, const uint16_t* pod_filter, int32_t n_filter,
                     int32_t* out_counts, kvb_pod_entry_t* out_entries, int64_t* out_cut) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    KVB_REQUIRE(n > 0 && keys, "no requestKeys provided for lookup");  // in_memory.go:110-112
    KVB_REQUIRE(out_counts && out_entries && out_cut, "NULL output");
    std::lock_guard<std::mutex> lk(idx->mu);
    DeviceGuard g(idx->device);
    const int32_t* cnt = nullptr;
    const uint32_t* ent = nullptr;
    // data.Get refreshes the outer LRU for every key that is found (in_memory.go:120): stamped by the kernel
    int rc = lookup_locked(idx, keys, n, pod_filter, n_filter, true, &cnt, &ent);
    if (rc) return rc;
    int64_t cut = n;
    for (int64_t i = 0; i < n; ++i) {
      if (cut < n || cnt[i] == -1) {  // after the cut nothing is looked at (in_memory.go:121-124 returns)
        out_counts[i] = -1;
        continue;
      }
      if (cnt[i] == -2) {  // present but empty: cannot occur (a key whose last pod leaves is removed), kept for parity
        cut = i;
        out_counts[i] = 0;
        continue;
      }
      out_counts[i] = cnt[i];
      for (int e = 0; e < cnt[i]; ++e) {
        const uint32_t v = ent[i * kMaxEnt + e];
        out_entries[i * kMaxEnt + e].pod = (uint16_t)(v & 0xffffu);
        out_entries[i * kMaxEnt + e].tier = (uint8_t)((v >> 16) & 0xffu);
        out_entries[i * kMaxEnt + e].speculative = (uint8_t)((v >> 24) & 1u);
      }
    }
    *out_cut = cut;
    return KVB_OK;
  });
}

#ifndef KVB_HOST_SIM
// memory a kernel can address in place: device memory, or pinned host memory (cudaHostAlloc / kvb_host_alloc /
// cudaHostRegister) through its device alias; nullptr for pageable host memory
static void* device_alias(const void* p) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
    cudaGetLastError();
    return nullptr;
  }
  if (a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeDevice) return a.devicePointer;
  return nullptr;
}

static int score_common(kvb_index* idx, const uint64_t* keys_host, const int64_t* key_off, int32_t n_prompts,
                        const uint32_t* tokens, const int64_t* prompt_off, const uint64_t* parents,
                        int32_t block_size, const uint8_t* extra, const int64_t* extra_off,
                        const uint16_t* pod_filter, int32_t n_filter, int32_t flags, int32_t* out_n,
                        uint16_t* out_pods, double* out_scores) {
  std::lock_guard<std::mutex> lk(idx->mu);
  DeviceGuard g(idx->device);
  int rc = idx->flush_locked();
  if (rc) return rc;
  const bool from_tokens = tokens != nullptr;
  const bool touch = (flags & KVB_SCORE_NO_TOUCH) == 0;
  const bool timing = (flags & KVB_SCORE_TIME_KERNELS) != 0;
  // ---- sizes
  int64_t total_keys = 0;
  if (from_tokens) {
    for (int32_t p = 0; p < n_prompts; ++p) {
      KVB_REQUIRE(prompt_off[p + 1] >= prompt_off[p], "prompt_off not monotonic at %d", p);
      total_keys += (prompt_off[p + 1] - prompt_off[p]) / block_size;
    }
  } else {
    total_keys = key_off[n_prompts] - key_off[0];
  }
  const int64_t total_tok = from_tokens ? prompt_off[n_prompts] - prompt_off[0] : 0;
  const int64_t extra_bytes = (from_tokens && extra_off) ? extra_off[total_keys] : 0;
  auto al = [](size_t x) { return (x + 255) & ~size_t(255); };
  // ---- one staging block, same offsets on the pinned host side and on the device:
  //      [koff | poff | parents | eoff | ext | host keys | filter bits]  -> ONE H2D;   [n | pods | scores]  <- kernel
  size_t o = 0;
  const size_t o_koff = o;   o += al(((size_t)n_prompts + 1) * 8);
  const size_t o_poff = o;   o += from_tokens ? al(((size_t)n_prompts + 1) * 8) : 0;
  const size_t o_par = o;    o += from_tokens ? al((size_t)n_prompts * 8) : 0;
  const size_t o_eoff = o;   o += (from_tokens && extra_off) ? al(((size_t)total_keys + 1) * 8) : 0;
  const size_t o_ext = o;    o += (from_tokens && extra_off) ? al((size_t)extra_bytes) : 0;
  const size_t o_hkeys = o;  o += from_tokens ? 0 : al((size_t)total_keys * 8);
  const size_t o_filt = o;   o += n_filter > 0 ? 2048 * sizeof(uint32_t) : 0;
  const size_t in_end = o;
  const size_t o_n = o;      o += al((size_t)n_prompts * 4);
  const size_t o_pods = o;   o += al((size_t)n_prompts * kMaxEnt * 2);
  const size_t o_sc = o;     o += al((size_t)n_prompts * kMaxEnt * 8);
  const size_t host_end = o;
  const size_t o_keys = o;   o += from_tokens ? al((size_t)total_keys * 8) : 0;  // device only: hashed keys
  const size_t o_tok = o;    o += from_tokens ? al((size_t)total_tok * 4) : 0;   // device only: copied tokens
  rc = idx->ensure_scratch(o, host_end);
  if (rc) return rc;
  uint8_t* H = idx->h_scratch;
  uint8_t* D = idx->d_scratch;
  cudaStream_t s = idx->stream;
  const uint32_t* filt = nullptr;
  bool filt_staged = false;
  rc = idx->set_filter(pod_filter, n_filter, H + o_filt, &filt_staged, &filt);
  if (rc) return rc;
  int64_t* h_koff = reinterpret_cast<int64_t*>(H + o_koff);
  if (from_tokens) {
    int64_t* h_poff = reinterpret_cast<int64_t*>(H + o_poff);
    h_koff[0] = 0;
    for (int32_t p = 0; p < n_prompts; ++p) {
      h_poff[p] = prompt_off[p] - prompt_off[0];
      h_koff[p + 1] = h_koff[p] + (prompt_off[p + 1] - prompt_off[p]) / block_size;
    }
    h_poff[n_prompts] = prompt_off[n_prompts] - prompt_off[0];
    std::memcpy(H + o_par, parents, (size_t)n_prompts * 8);
    if (extra_off) {
      std::memcpy(H + o_eoff, extra_off, ((size_t)total_keys + 1) * 8);
      if (extra_bytes) std::memcpy(H + o_ext, extra, (size_t)extra_bytes);
    }
  } else {
    for (int32_t p = 0; p <= n_prompts; ++p) h_koff[p] = key_off[p] - key_off[0];
    if (total_keys > 0) std::memcpy(H + o_hkeys, keys_host + key_off[0], (size_t)total_keys * 8);
  }
  // results land where the caller wants them when that memory is pinned (no D2H copy, no memcpy); otherwise in the
  // pinned staging block through its device alias
  uint8_t* Hd = idx->h_scratch_dev;
  // KVB_SCORE_PINNED_IO: the caller vouches that tokens and outputs are pinned (kvb_host_alloc / cudaHostAlloc) — with
  // unified addressing a kernel uses the same address, and four pointer queries (~1 us each) leave the call
  const bool pinned_io = (flags & KVB_SCORE_PINNED_IO) != 0;
  int32_t* k_n = pinned_io ? out_n : static_cast<int32_t*>(device_alias(out_n));
  uint16_t* k_pods = pinned_io ? out_pods : static_cast<uint16_t*>(device_alias(out_pods));
  double* k_sc = pinned_io ? out_scores : static_cast<double*>(device_alias(out_scores));
  const bool direct_out = k_n && k_pods && k_sc;
  if (!direct_out) {
    k_n = reinterpret_cast<int32_t*>(Hd + o_n);
    k_pods = reinterpret_cast<uint16_t*>(Hd + o_pods);
    k_sc = reinterpret_cast<double*>(Hd + o_sc);
  }
  unsigned long long stamp_base = 0ull;
  if (touch) {
    stamp_base = idx->seq;
    idx->seq += (unsigned long long)total_keys;
  }
  // the small arrays: one copy — or none at all for a handful of prompts, where the kernel reads the pinned staging
  // block in place (one PCIe round trip instead of a copy operation ahead of the launch)
  const bool small_in_place = from_tokens && n_prompts <= 64 && !extra_off && (flags & KVB_SCORE_COPY_TOKENS) == 0;
  const uint8_t* Din = small_in_place ? Hd : D;  // where the kernels read koff / poff / parents
  const size_t small_end = (n_filter > 0) ? o_filt : in_end;  // the filter bitmap was copied by set_filter (if it changed)
  if (timing) KVB_CUDA_TRY(cudaEventRecord(idx->ev_a, s));
  if (!small_in_place)
    KVB_CUDA_TRY(cudaMemcpyAsync(D + o_koff, H + o_koff, small_end - o_koff, cudaMemcpyHostToDevice, s));
  const uint64_t* d_keys = reinterpret_cast<const uint64_t*>(D + (from_tokens ? o_keys : o_hkeys));
  bool scored = false, watch_flag = false;
  if (from_tokens && total_keys > 0) {
    // tokens: pinned buffers (kvb_host_alloc / cudaHostAlloc / registered) are read IN PLACE by the stager warps — the
    // PCIe transfer overlaps the hash chains instead of preceding them; pageable buffers are copied (staged by the driver)
    const uint32_t* tok_dev = pinned_io ? tokens + prompt_off[0]
                                        : static_cast<const uint32_t*>(device_alias(tokens + prompt_off[0]));
    if (tok_dev == nullptr || (flags & KVB_SCORE_COPY_TOKENS) != 0) {
      KVB_CUDA_TRY(cudaMemcpyAsync(D + o_tok, tokens + prompt_off[0], (size_t)total_tok * 4, cudaMemcpyHostToDevice, s));
      tok_dev = reinterpret_cast<const uint32_t*>(D + o_tok);
    }
    ChainArgs a{};
    a.tokens = tok_dev;
    a.tokens_lo = tok_dev;  // 16 B granules are read only inside [lo, hi): nothing outside the caller's array is touched
    a.tokens_hi = tok_dev + total_tok;
    a.single = (n_prompts == 1 && !extra_off) ? 1 : 0;
    a.single_tokens = total_tok;
    a.single_parent = parents[0];
    a.prompt_off = reinterpret_cast<const int64_t*>(Din + o_poff);
    a.parents = reinterpret_cast<const uint64_t*>(Din + o_par);
    a.extra = extra_off ? D + o_ext : nullptr;
    a.extra_off = extra_off ? reinterpret_cast<const int64_t*>(D + o_eoff) : nullptr;
    a.out_keys = nullptr;
    a.key_off = reinterpret_cast<const int64_t*>(Din + o_koff);
    a.table = idx->table;
    a.mask = idx->slots - 1;
    a.filter_bits = filt;
    a.tier_w = idx->tier_w;
    a.out_n = k_n;
    a.out_pods = k_pods;
    a.out_scores = k_sc;
    a.ts = touch ? idx->ts : nullptr;
    a.stamp_base = stamp_base;
    a.score_min_batch = n_prompts <= 256 ? 4 : 32;
    const bool fuse = n_prompts <= 1536 && (flags & KVB_SCORE_TWO_KERNELS) == 0;
    if (fuse && !timing) {  // completion word: the last prompt to finish writes this call's number to pinned memory
      a.done_counter = idx->d_done;
      a.done_target = (unsigned)n_prompts;
      a.done_flag_host = idx->h_done;
      a.done_value = ++idx->done_seq;
    }
    // a handful of prompts: the table kernel (token bytes off the chain, any block size); else the chain kernel
    int spec_rc = KVB_OK;
    if (fuse && launch_spec_score(a, n_prompts, block_size, total_keys, s, &spec_rc,
                                  reinterpret_cast<const int64_t*>(H + o_poff), h_koff,
                                  reinterpret_cast<const uint64_t*>(H + o_par), idx->spec)) {
      if (spec_rc) return spec_rc;
      scored = true;
      watch_flag = a.done_counter != nullptr;
    } else if (fuse && launch_chain_score(a, n_prompts, block_size, s)) {
      KVB_CUDA_TRY(cudaGetLastError());
      scored = true;  // ONE launch did tokens -> keys -> lookup -> scores
      watch_flag = a.done_counter != nullptr;
    } else {
      rc = launch_hash_blocks(tok_dev, a.prompt_off, a.parents, n_prompts, block_size, a.extra, a.extra_off,
                              reinterpret_cast<uint64_t*>(D + o_keys), a.key_off, s, total_keys,
                              reinterpret_cast<const int64_t*>(H + o_poff), h_koff,
                              reinterpret_cast<const uint64_t*>(H + o_par), idx->spec);
      if (rc) return rc;
    }
  }
  if (timing) KVB_CUDA_TRY(cudaEventRecord(idx->ev_b, s));
  if (!scored) {
    const int64_t grid = ((int64_t)n_prompts + kScoreWarps - 1) / kScoreWarps;
    index_score_kernel<<<(unsigned)grid, kScoreWarps * 32, 0, s>>>(
        idx->table, idx->slots - 1, d_keys, reinterpret_cast<const int64_t*>(Din + o_koff), n_prompts, filt, idx->tier_w,
        k_n, k_pods, k_sc, touch ? idx->ts : nullptr, stamp_base);
    KVB_CUDA_TRY(cudaGetLastError());
    count_launch();
  }
  if (timing) KVB_CUDA_TRY(cudaEventRecord(idx->ev_c, s));
  bool finished = false;
  if (watch_flag) {
    // the kernel's last act is a store of done_seq to pinned memory (after a system fence behind every result): watching
    // that word costs about a microsecond, a stream synchronisation several.  Bounded: a faulting kernel never writes it.
    const volatile unsigned long long* flag = idx->h_done;
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned spins = 0;; ++spins) {
      if (*flag == idx->done_seq) {
        finished = true;
        break;
      }
      if ((spins & 1023u) == 1023u &&
          std::chrono::duration_cast<std::chrono::microseconds>(std::chrono::steady_clock::now() - t0).count() > 5000)
        break;
    }
  }
  if (!finished) KVB_CUDA_TRY(cudaStreamSynchronize(s));
  if (!direct_out) {
    std::memcpy(out_n, H + o_n, (size_t)n_prompts * 4);
    std::memcpy(out_pods, H + o_pods, (size_t)n_prompts * kMaxEnt * 2);
    std::memcpy(out_scores, H + o_sc, (size_t)n_prompts * kMaxEnt * 8);
  }
  if (timing) {
    float ab = 0.f, bc = 0.f;
    cudaEventElapsedTime(&ab, idx->ev_a, idx->ev_b);
    cudaEventElapsedTime(&bc, idx->ev_b, idx->ev_c);
    idx->last_hash_us = ab * 1e3f;  // staging copies + hash kernel
    idx->last_score_us = bc * 1e3f;
  }
  return KVB_OK;
}

int kvb_index_score_batch(kvb_index_t* idx, const uint64_t* keys, const int64_t* key_off, int32_t n_prompts,
                          const uint16_t* pod_filter, int32_t n_filter, int32_t flags, int32_t* out_n,
                          uint16_t* out_pods, double* out_scores) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    KVB_REQUIRE(n_prompts >= 0, "negative prompt count");
    if (n_prompts == 0) return KVB_OK;
    KVB_REQUIRE(key_off && out_n && out_pods && out_scores, "NULL argument");
    KVB_REQUIRE(keys || key_off[n_prompts] == key_off[0], "keys is NULL");
    return score_common(idx, keys, key_off, n_prompts, nullptr, nullptr, nullptr, 0, nullptr, nullptr, pod_filter,
                        n_filter, flags, out_n, out_pods, out_scores);
  });
}

int kvb_index_score_tokens_batch(kvb_index_t* idx, const uint32_t* tokens, const int64_t* prompt_off,
                                 const uint64_t* parents, int32_t n_prompts, int32_t block_size, const uint8_t* extra,
                                 const int64_t* extra_off, const uint16_t* pod_filter, int32_t n_filter,
                                 int32_t flags, int32_t* out_n, uint16_t* out_pods, double* out_scores) {
  return kvb::guarded([&]() -> int {
    KVB_REQUIRE(idx != nullptr, "index is NULL");
    KVB_REQUIRE(block_size > 0, "blockSize must be greater than 0, got %d", block_size);
    KVB_REQUIRE(n_prompts >= 0, "negative prompt count");
    if (n_prompts == 0) return KVB_OK;
    KVB_REQUIRE(tokens && prompt_off && parents && out_n && out_pods && out_scores, "NULL argument");
    return score_common(idx, nullptr, nullptr, n_prompts, tokens, prompt_off, parents, block_size, extra, extra_off,
                        pod_filter, n_filter, flags, out_n, out_pods, out_scores);
  });
}
#endif  // !KVB_HOST_SIM

}  // extern "C"
