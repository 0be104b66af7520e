/* kvb.h — C ABI of libkvb.so, the B200-native (sm_100a) KV-block hot path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / C++ types.
 * Each group of entry points names the reference interface it replaces
 * (paths relative to llm-d/llm-d-kv-cache @ 82d31d1).  INTEGRATION.md shows the
 * reference-side bindings (cgo for the Go indexer, ctypes for the vLLM plugin).
 *
 * Conventions
 *   - every function returning int returns KVB_OK (0) or a negative KVB_ERR_*;
 *     kvb_last_error() gives the message for the calling thread.  No exceptions
 *     cross this boundary (reference: tasks catch everything and return bool,
 *     csrc/storage/storage_offload.cpp:338-347,405-411).
 *   - "stream" arguments are cudaStream_t passed as void*; NULL = legacy default stream.
 *   - block ids are int64 (reference: std::vector<int64_t>, storage_offload.hpp:104-109).
 *   - there is NO CPU fallback: every compute entry point fails with KVB_ERR_CUDA
 *     when no sm_100 device is usable.
 *   - environment switches (diagnostics and A/B runs, never needed for correctness):
 *       KVB_HASH_KERNEL=lanes   hash with the lane-per-prompt kernels at every batch size (read per call)
 *       KVB_HASH_KERNEL=wpc     hash with the warp-per-prompt kernel at every batch size it supports (the default up to 1536 prompts)
 *       KVB_HASH_KERNEL=chain   hash with round 2's chain kernel in its hash-only form (it is the fused scoring launch's kernel)
 *       KVB_HASH_KERNEL=spec    the table kernel for every batch it can take (<= 64 prompts, <= 16384 keys; default: <= 32 prompts)
 *       KVB_HASH_SPEC=0         never pick the table kernel;  KVB_SPEC_SCORE_BATCH=1..32  keys its scorer warp waits for
 *       KVB_INDEX_PLAN=0        index at capacity: replay batches on one thread instead of planning their evictions
 *       KVB_INDEX_SCAN_MAX_SLOTS=n   largest table the one-thread replay may scan for its oldest key when the LRU order array
 *                               runs out mid-batch (default 65536; larger tables stop, rebuild the order array and resume)
 *       KVB_HASH_MERGED=0|1     chain kernel: vote-free first two bits off / on (default: on up to 512 prompts)
 *       KVB_CHAIN_FETCH=128x2|256x2|256x4|128x6   chain kernel: token chunk size x chunks in flight
 *       KVB_HASH_ONE_WARP=1     hash with the one-warp lane kernel (read once)
 *       KVB_NO_NUMA_BIND=1      do not bind engine threads / arena to the GPU's NUMA node
 *       KVB_FILE_WRITE=pwrite|mmap   file tier: force one write path (default: pwrite per worker, a shared mapping written by
 *                                    KVB_FILE_LONE_PARTS helper threads (8) when a store is alone in the queue)
 *       KVB_FILE_SPREAD=1       file tier: every second worker runs on the other NUMA node's CPUs
 */
#ifndef KVB_H_
#define KVB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KVB_ABI_VERSION 5

#define KVB_OK 0
#define KVB_ERR_INVALID (-1)   /* bad argument */
#define KVB_ERR_CUDA (-2)      /* CUDA runtime / no device */
#define KVB_ERR_NOMEM (-3)     /* host or device allocation failed / arena full */
#define KVB_ERR_NOTFOUND (-4)  /* unknown key / job / file */
#define KVB_ERR_IO (-5)        /* file tier I/O */
#define KVB_ERR_UNSUPPORTED (-6)

int kvb_abi_version(void);
const char* kvb_last_error(void);
int kvb_device_count(void);
/* pinned (page-locked, portable) host memory: buffers allocated here are read/written by the copy engines in place,
 * pageable buffers are staged through an internal pinned scratch first */
int kvb_host_alloc(size_t bytes, void** out);
int kvb_host_free(void* p);
/* the same with the backing chosen: KVB_HOST_ALLOC_THP = anonymous memory advised to transparent huge pages, first-touched
 * on the GPU's NUMA node and registered with CUDA (fewer, larger DMA translations; measured beside the default in the
 * bench's PCIe probe) */
#define KVB_HOST_ALLOC_DEFAULT 0
#define KVB_HOST_ALLOC_THP 1
int kvb_host_alloc_mode(size_t bytes, int mode, void** out);

/* ------------------------------------------------------------------------------------------
 * 1. Paged-KV pool + gather / scatter  (HBM <-> packed HBM)
 *    replaces TensorCopier::copy_blocks (csrc/storage/tensor_copier.cu:50-109) and
 *    copy_blocks_kernel (tensor_copier_kernels.cu:54-143).
 *    Pool = T canonical KV tensors, each (num_blocks, frag_bytes) bytes with row stride
 *    block_stride_bytes (tensor_copier.cu:39: frag = stride(0)*element_size).  Tensors are
 *    BORROWED (owned by the caller / vLLM, tensor_copier.hpp:41).
 *    Packed layout = [block][tensor][fragment] (tensor_copier.cu:73-96).
 * ------------------------------------------------------------------------------------------ */
typedef struct kvb_pool kvb_pool_t;

/* copy-kernel variants (flags argument of gather/scatter; 0 = library default) */
#define KVB_COPY_DEFAULT 0
#define KVB_COPY_LDG 1  /* 16 B vector LDG/STG, unrolled, persistent grid */
#define KVB_COPY_BULK 2 /* TMA bulk copies (cp.async.bulk) staged through shared memory */

int kvb_pool_create(int device, const void* const* tensor_ptrs, int32_t num_tensors, int64_t num_blocks,
                    int64_t frag_bytes, int64_t block_stride_bytes, kvb_pool_t** out);
void kvb_pool_destroy(kvb_pool_t* pool);
int64_t kvb_pool_block_bytes(const kvb_pool_t* pool); /* T * frag_bytes */
/* declare that the pool's tensors live on another GPU (peer-enabled or CUDA-IPC mapped): kvb_migrate_blocks then
 * defaults to the mover tuned for NVLink stores.  Auto-detected when the driver reports the owning device. */
int kvb_pool_mark_peer(kvb_pool_t* pool, int is_peer);

/* block_ids: HOST array of n ids.  packed: DEVICE (or device-mapped / peer) buffer of n*T*frag bytes. */
int kvb_gather_blocks(kvb_pool_t* pool, const int64_t* block_ids, int64_t n, void* packed, void* stream, int flags);
int kvb_scatter_blocks(kvb_pool_t* pool, const int64_t* block_ids, int64_t n, const void* packed, void* stream,
                       int flags);
/* same, block ids already resident on the device (no upload; used by the timed bench loop) */
int kvb_gather_blocks_dev(kvb_pool_t* pool, const int64_t* block_ids_dev, int64_t n, void* packed, void* stream,
                          int flags);
int kvb_scatter_blocks_dev(kvb_pool_t* pool, const int64_t* block_ids_dev, int64_t n, const void* packed,
                           void* stream, int flags);
/* number of kernels launched by this library in this process (bench "gpu_launches") */
int64_t kvb_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * 2. Offload engine (save_blocks / load_blocks)
 *    replaces storage_offload.StorageOffloadEngine (csrc/storage/storage_offload_bindings.cpp:25-94;
 *    storage_offload.cpp:57-77 ctor, :249 async_store_gpu_blocks, :362 async_load_gpu_blocks,
 *    :185 get_finished, :214 wait_job) — the StorageEngine Protocol of llmd_fs_backend/worker.py:36-52.
 * ------------------------------------------------------------------------------------------ */
typedef struct kvb_engine kvb_engine_t;

#define KVB_TIER_FILE 0       /* reference on-disk format (file_io.cpp:50-225): tail-aligned, full-size .bin */
#define KVB_TIER_HOST_ARENA 1 /* pinned host DRAM arena keyed by the same path strings */

typedef struct kvb_engine_opts {
  int32_t io_threads;              /* file-tier worker threads (reference: io_threads) */
  int32_t gpu_blocks_per_file;     /* reference: gpu_blocks_per_file */
  int32_t read_preferring_workers; /* reference: read_preferring_workers (thread_pool.cpp:47-57) */
  float max_write_queued_seconds;  /* reference: dynamic write-queue limit, 0 = off (storage_offload.cpp:96-105) */
  int32_t tier;                    /* KVB_TIER_* */
  int32_t copy_flags;              /* KVB_COPY_* */
  int64_t host_arena_bytes;        /* KVB_TIER_HOST_ARENA capacity */
  int64_t chunk_bytes;             /* bytes gathered per kernel launch = packed HBM staging per worker (0 = 64 MiB);
                                      a chunk always holds whole files */
  int32_t direct_host_io;          /* 1 = the gather/scatter kernels read/write the pinned host buffers directly
                                      (fused gather+D2H / H2D+scatter, no HBM staging, no cudaMemcpy); 0 = staged */
  int32_t strict_load_errors;      /* file tier only.  0 = reference behaviour: a FILE that is missing / short / unreadable is
                                      logged and the job still reports ok (storage_offload.cpp:378-383); 1 = report ok=0.
                                      Anything else that kept pages from being restored — a host-arena miss (the arena's own
                                      LRU dropped the entry), a CUDA error, a failed launch — ALWAYS reports ok=0.  Worker
                                      resources are allocated inside kvb_engine_create: if io_threads x chunk_bytes does not
                                      fit, create fails with KVB_ERR_NOMEM */
  int32_t gds_mode;                /* KVB_GDS_* bits, file tier only: reference gds_mode (gds_file_io.cpp:425-446).  Files
                                      are then the reference's GDS format (head-aligned, n x block_bytes long) moved by
                                      cuFile between the file and the packed HBM chunk, ONE call per file.  Falls back to
                                      the CPU-staged path when libcufile cannot be loaded (storage_offload.cpp:129-134) */
  int32_t arena_alloc_mode;        /* KVB_HOST_ALLOC_* backing of the host arena (0 = cudaHostAlloc, the default) */
} kvb_engine_opts_t;

#define KVB_GDS_DISABLED 0
#define KVB_GDS_READ 1   /* loads through cuFileRead */
#define KVB_GDS_WRITE 2  /* stores through cuFileWrite */
#define KVB_GDS_BOUNCE 4 /* reference "bb_*" modes; same data path here (the packed chunk is the registered buffer) */

void kvb_engine_default_opts(kvb_engine_opts_t* opts);
int kvb_engine_create(kvb_pool_t* pool, const kvb_engine_opts_t* opts, kvb_engine_t** out);
void kvb_engine_destroy(kvb_engine_t* eng);

/* files[i] receives / provides block_ids[file_off[i] .. file_off[i+1]) ; file_off has n_files+1 entries.
 * caller_stream: the stream the KV was produced on; the copy is ordered after it
 * (storage_offload.cpp:259-265).  Submit only — returns immediately. */
int kvb_engine_store(kvb_engine_t* eng, int64_t job_id, int32_t n_files, const char* const* files,
                     const int64_t* block_ids, const int64_t* file_off, void* caller_stream);
int kvb_engine_load(kvb_engine_t* eng, int64_t job_id, int32_t n_files, const char* const* files,
                    const int64_t* block_ids, const int64_t* file_off, void* caller_stream);
/* get_finished(): drains up to cap finished jobs; returns count (>=0) or error (<0). */
int kvb_engine_poll(kvb_engine_t* eng, int64_t* job_ids, int32_t* ok, int32_t cap);
/* wait_job(): cancels still-queued file tasks of the job, then blocks until it is finished. */
int kvb_engine_wait(kvb_engine_t* eng, int64_t job_id);
/* manager-side lookup (llmd_fs_backend/manager.py:43-53): 1 if the file/arena entry exists */
int kvb_engine_exists(kvb_engine_t* eng, const char* file);
/* SharedStorageOffloadingManager.lookup in ONE call (manager.py:43-53): the number of CONSECUTIVE entries of files[]
 * from the start that exist — the loop stops at the first miss, like the reference's.  Arena tier: hash-map probes
 * under one lock; file tier: one statx per file, nothing else (no Python, no per-block FFI crossing). */
int kvb_engine_lookup_prefix(kvb_engine_t* eng, int32_t n_files, const char* const* files, int32_t* out_hits);
/* the same with the file names built inside the library from the low 64 bits of the block hashes
 * (FileMapper.get_file_name, file_mapper.py:69-87: <base_path>/<hhh>/<hh>/<016x>.bin): 8 bytes per block cross the
 * boundary instead of a path string */
int kvb_engine_lookup_prefix_hashes(kvb_engine_t* eng, const char* base_path, const uint64_t* hashes, int32_t n,
                                    int32_t* out_hits);
/* drop every host-arena entry (test / bench helper) */
int kvb_engine_arena_clear(kvb_engine_t* eng);

typedef struct kvb_engine_stats {
  int64_t bytes_stored, bytes_loaded;     /* payload bytes moved */
  int64_t files_stored, files_loaded;
  int64_t files_skipped_existing;         /* storage_offload.cpp:299-304 */
  int64_t writes_dropped;                 /* storage_offload.cpp:272-288 */
  int64_t load_failures;                  /* reported as ok=0 (reference swallows them, :381-383) */
  int64_t kernels_launched;
  int64_t h2d_bytes, d2h_bytes;
} kvb_engine_stats_t;
int kvb_engine_get_stats(kvb_engine_t* eng, kvb_engine_stats_t* out);

/* ------------------------------------------------------------------------------------------
 * 3. Block-key hashing
 *    replaces kvblock.TokenProcessor (pkg/kvcache/kvblock/token_processor.go:55-69):
 *    key_i = FNV64a(CBORcanonical([parent, chunk_i, extra_i])) chained (:123-153).
 * ------------------------------------------------------------------------------------------ */
uint64_t kvb_fnv64a(const void* data, size_t len); /* seed hash, token_processor.go:90-95 (host, setup only) */
/* getInitHash (token_processor.go:109-111) = H(seed_hash, nil, model_name); computed on the device */
int kvb_init_hash(int device, uint64_t seed_hash, const char* model_name, size_t model_len, uint64_t* out);

/* Batched TokensToKVBlockKeys (token_processor.go:177-205).
 *   tokens      HOST  uint32, all prompts concatenated
 *   prompt_off  HOST  int64[n_prompts+1] token offsets
 *   parents     HOST  uint64[n_prompts]: parentKey if != 0 else the init hash (:181-186)
 *   extra / extra_off  optional per-BLOCK trailing CBOR item (multimodal taint, :146-148):
 *                      extra_off int64[total_blocks+1] into extra bytes; NULL => every block is text (0xf6).
 *                      A zero-length slice also means 0xf6.
 *   out_keys    HOST  uint64[>= total_blocks]; out_key_off HOST int64[n_prompts+1]
 * Only full blocks produce keys (chunkTokens, :161-174). */
int kvb_hash_token_blocks(int device, const uint32_t* tokens, const int64_t* prompt_off, const uint64_t* parents,
                          int32_t n_prompts, int32_t block_size, const uint8_t* extra, const int64_t* extra_off,
                          uint64_t* out_keys, int64_t* out_key_off, void* stream);
/* device-resident variant: every pointer is a DEVICE pointer, key_off precomputed; no host sync.
 * total_keys = key_off[n_prompts] if the caller knows it (small batches then use the table kernel), else -1 */
int kvb_hash_token_blocks_dev(int device, const uint32_t* tokens, const int64_t* prompt_off, const uint64_t* parents,
                              int32_t n_prompts, int32_t block_size, const uint8_t* extra, const int64_t* extra_off,
                              uint64_t* out_keys, const int64_t* key_off, int64_t total_keys, void* stream);

/* ------------------------------------------------------------------------------------------
 * 4. Block index + longest-prefix scorer
 *    replaces kvblock.Index (pkg/kvcache/kvblock/index.go:120-149; in_memory.go:107-304) and
 *    LongestPrefixScorer.Score (pkg/kvcache/kvblock_scorer.go:106-154).
 *    Pod identifiers and device tiers are interned to dense ids by the host shim.
 * ------------------------------------------------------------------------------------------ */
typedef struct kvb_index kvb_index_t;

typedef struct kvb_pod_entry { /* kvblock.PodEntry, index.go:176-183 */
  uint16_t pod;                /* interned PodIdentifier */
  uint8_t tier;                /* interned DeviceTier */
  uint8_t speculative;         /* 0 / 1 */
} kvb_pod_entry_t;

#define KVB_INDEX_MAX_PODS_PER_KEY 13 /* entries that fit one 64 B bucket */
#define KVB_KEY_ENGINE 0              /* index.go:155-161 */
#define KVB_KEY_REQUEST 1

/* max_keys = InMemoryIndexConfig.Size, pods_per_key = PodCacheSize (in_memory.go:40-45);
 * table_slots = device buckets (power of two, 0 = auto from expected_keys). */
int kvb_index_create(int device, int64_t max_keys, int32_t pods_per_key, int64_t expected_keys, kvb_index_t** out);
void kvb_index_destroy(kvb_index_t* idx);
int kvb_index_set_tier_weight(kvb_index_t* idx, uint8_t tier, double weight, int known);

int kvb_index_add(kvb_index_t* idx, const uint64_t* engine_keys, int64_t n_engine, int has_engine_keys,
                  const uint64_t* request_keys, int64_t n_request, const kvb_pod_entry_t* entries, int32_t n_entries);
int kvb_index_evict(kvb_index_t* idx, uint64_t key, int key_type, const kvb_pod_entry_t* entries, int32_t n_entries);
int kvb_index_get_request_key(kvb_index_t* idx, uint64_t engine_key, uint64_t* out);
int64_t kvb_index_num_keys(kvb_index_t* idx);
/* KV-event ingest, the writer side of the index: Pool.processEventBatch (pkg/kvevents/pool.go:253-398) for a DECODED batch
 * in one call.  Events of one `stream` (the pod) are applied in order, streams are independent (the reference shards pods
 * over parallel workers, pool.go:154-166).  Per round the library resolves the parents of the BlockStored events through the
 * engine-key map (GetRequestKey; an unknown parent drops the event, pool.go:284-294), hashes them in ONE device launch and adds
 * them; BlockRemoved events evict by engine key (pool.go:379-386).  Text-only events: multimodal extras go through
 * kvb_hash_token_blocks + kvb_index_add.  *out_skipped = events the reference would log and skip. */
#define KVB_EVENT_BLOCK_STORED 0
#define KVB_EVENT_BLOCK_REMOVED 1
#define KVB_EVENT_OTHER 2 /* AllBlocksCleared / unknown: ignored, as in the reference (pool.go:388-395) */
#define KVB_EVENT_POD_CLEARED 3 /* remove entry.pod's entries of entry.tier (kvb_index_remove_pods; opt-in AllBlocksCleared).
                                   Applied at its place among the round's non-stored events: what is queued goes first */
typedef struct kvb_kv_event {
  int32_t type;               /* KVB_EVENT_* */
  int32_t stream;             /* ordering domain: the pod */
  int64_t token_off, n_tokens;            /* into tokens[] (BlockStored) */
  int64_t engine_key_off, n_engine_keys;  /* into engine_keys[]: BlockStored.BlockHashes / BlockRemoved.BlockHashes */
  uint64_t parent_engine_key; /* BlockStored.ParentHash, 0 = none */
  uint64_t root_hash;         /* getInitHash of the event's model or LoRA name (pool.go:271-274): parent of a parentless event */
  kvb_pod_entry_t entry;      /* the pod and the event's device tier */
  int32_t pad;
} kvb_kv_event_t;
int kvb_index_ingest_events(kvb_index_t* idx, const kvb_kv_event_t* events, int32_t n_events, const uint32_t* tokens,
                            const uint64_t* engine_keys, int32_t block_size, int32_t* out_skipped);

/* Remove every entry of `pods` (interned ids, n_pods >= 1) from every key; tiers == NULL / n_tiers == 0: every tier,
 * otherwise an entry goes only if its tier is listed too.  The speculative bit is not looked at.  No reference
 * counterpart (pool.go:388-395 ignores AllBlocksCleared): one device sweep over the whole table, since only the table
 * knows which request keys hold a pod.
 *   - surviving entries keep their inner-LRU order; a key left empty is deleted (in_memory.go:281-292)
 *   - no recency stamp changes (a sequence of Evict calls would refresh every key it touches); the engine-key map is
 *     untouched, as Evict(RequestKey) leaves it
 *   - queued Add / Evict ops are applied first, ops queued later come after: the result is that of call order
 *   - ids never interned simply match nothing
 * out_entries_removed / out_keys_deleted may be NULL. */
int kvb_index_remove_pods(kvb_index_t* idx, const uint16_t* pods, int32_t n_pods, const uint8_t* tiers, int32_t n_tiers,
                          int64_t* out_entries_removed, int64_t* out_keys_deleted);

/* apply the queued Add / Evict operations to the device table and wait for it (reads do this implicitly) */
int kvb_index_flush(kvb_index_t* idx, void* stream);

/* The index is device-authoritative: buckets, per-key pod lists and the outer LRU order (one recency stamp per slot)
 * live in HBM and are mutated by kernels; the host keeps only the engine-key map.  Counters for tests and the bench. */
typedef struct kvb_index_stats {
  int64_t live_keys, tombstones, table_slots, engine_keys;
  int64_t ops_applied;        /* Add / Evict records applied on the device */
  int64_t flushes_parallel;   /* sorted, one thread per distinct key */
  int64_t flushes_sequential; /* one thread in the reference's order (tiny batches; at capacity, batches whose eviction
                                 plan did not settle) */
  int64_t flushes_planned;    /* parallel flushes at capacity: LRU victims planned up front, same result as in order */
  int64_t plan_fallbacks;     /* planned flushes that had to be replayed sequentially */
  int64_t replay_resumes;     /* sequential replays that stopped for a fresh LRU order array and resumed (large tables) */
  int64_t rehashes;           /* device-side table growth / tombstone purge */
  int64_t lru_evictions;      /* keys dropped because the index held `max_keys` (in_memory.go:197) */
  int64_t order_builds, order_stale_skipped, order_scans; /* LRU order array: sorts, stale records skipped, fallbacks */
  float last_hash_us, last_score_us; /* device time of the last scoring call made with KVB_SCORE_TIME_KERNELS: copies +
                                        hash kernel and score kernel (two-kernel mode), or the whole fused launch in
                                        last_hash_us and 0 in last_score_us */
} kvb_index_stats_t;
int kvb_index_get_stats(kvb_index_t* idx, kvb_index_stats_t* out);

/* Lookup (in_memory.go:107-148) on the device.  pod_filter: interned ids (n_filter = 0 => all pods).
 * out_counts[i]: -1 key absent, otherwise number of entries written to
 * out_entries[i*KVB_INDEX_MAX_PODS_PER_KEY ...] after filtering.  *out_cut = index of the first
 * present-but-empty key (lookup stops there), or n if none. */
int kvb_index_lookup(kvb_index_t* idx, const uint64_t* keys, int64_t n, const uint16_t* pod_filter, int32_t n_filter,
                     int32_t* out_counts, kvb_pod_entry_t* out_entries, int64_t* out_cut);

/* Batched Lookup + Score for many prompts: keys HOST uint64 flat, key_off HOST int64[n_prompts+1].
 * Per prompt up to KVB_INDEX_MAX_PODS_PER_KEY (pod, score) pairs: out_n[p] pairs in
 * out_pods/out_scores[p*KVB_INDEX_MAX_PODS_PER_KEY ...].  Scores are float64 sums in key order. */
/* flags.  Every found key's outer-LRU recency is refreshed BY DEFAULT, as Lookup's data.Get does (in_memory.go:120):
 * the scoring kernel stamps the slot, the host does nothing. */
#define KVB_SCORE_TOUCH_LRU 1    /* accepted for source compatibility; this is the default now */
#define KVB_SCORE_NO_TOUCH 2     /* opt out: read-only scoring (e.g. what-if queries that must not disturb eviction order) */
#define KVB_SCORE_TIME_KERNELS 4 /* record CUDA events around the kernels; read them with kvb_index_get_stats */
#define KVB_SCORE_COPY_TOKENS 8  /* A/B: copy pinned token buffers to HBM first instead of reading them in place */
#define KVB_SCORE_TWO_KERNELS 16 /* A/B: hash kernel + score kernel instead of the fused tokens -> scores launch */
#define KVB_SCORE_PINNED_IO 32   /* the caller vouches that tokens AND the three output arrays are pinned host memory
                                    (kvb_host_alloc): they are read / written in place without asking the driver */
int kvb_index_score_batch(kvb_index_t* idx, const uint64_t* keys, const int64_t* key_off, int32_t n_prompts,
                          const uint16_t* pod_filter, int32_t n_filter, int32_t flags, int32_t* out_n,
                          uint16_t* out_pods, double* out_scores);
/* Fused Indexer.ScoreTokens (pkg/kvcache/indexer.go:239-304) for a batch: tokens -> keys -> lookup -> score,
 * all on the device; only tokens go in and (pod, score) pairs come out.  Arguments as in
 * kvb_hash_token_blocks + kvb_index_score_batch. */
int kvb_index_score_tokens_batch(kvb_index_t* idx, const uint32_t* tokens, const int64_t* prompt_off,
                                 const uint64_t* parents, int32_t n_prompts, int32_t block_size, const uint8_t* extra,
                                 const int64_t* extra_off, const uint16_t* pod_filter, int32_t n_filter,
                                 int32_t flags, int32_t* out_n, uint16_t* out_pods, double* out_scores);
/* debug: the entries of one key (oldest->newest) read back from the device WITHOUT refreshing its recency;
 * returns the count or -1 if absent */
int kvb_index_host_peek(kvb_index_t* idx, uint64_t request_key, kvb_pod_entry_t* out_entries, int32_t cap);

/* ------------------------------------------------------------------------------------------
 * 5. Cross-GPU block migration (no reference counterpart; data layout of section 1)
 *    One process per GPU: the destination exports its pool over CUDA IPC, the source maps it and
 *    a single kernel reads source pages and writes destination pages over NVLink.
 * ------------------------------------------------------------------------------------------ */
#define KVB_IPC_HANDLE_BYTES 64
typedef struct kvb_ipc_mem {
  uint8_t handle[KVB_IPC_HANDLE_BYTES]; /* cudaIpcMemHandle_t of the allocation base */
  int64_t offset;                       /* pointer - allocation base */
} kvb_ipc_mem_t;

int kvb_ipc_export(int device, const void* dev_ptr, kvb_ipc_mem_t* out);
int kvb_ipc_import(int device, const kvb_ipc_mem_t* mem, void** out_ptr);
int kvb_ipc_close(int device, void* imported_ptr, int64_t offset);
int kvb_enable_peer_access(int device, int peer_device);

/* src pool pages src_ids[i] -> dst pool pages dst_ids[i]; dst pool may live on a peer GPU
 * (tensor pointers peer-mapped or IPC-imported).  Runs on src->device. */
int kvb_migrate_blocks(kvb_pool_t* src, kvb_pool_t* dst, const int64_t* src_ids, const int64_t* dst_ids, int64_t n,
                       void* stream, int flags);

#ifdef __cplusplus
}
#endif
#endif /* KVB_H_ */
