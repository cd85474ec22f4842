/*
 * vega_b200.h — C ABI of libvega_b200.so: a B200-native (sm_100a) shuffle + aggregation
 * engine that drops in behind rajasekarv/vega's RDD operator API for the path
 *   group_by_key / reduce_by_key / join (cogroup) / partition_by_key  (+ sort_by_key, new).
 *
 * The reference has no FFI today (SURVEY.md F4); these entry points are what a thin Rust
 * `extern "C"` shim binds at the four trait seams (INTEGRATION.md shows the shim):
 *
 *   vb_shuffle_create      <- ShuffleDependency::new              src/dependency.rs:133-149
 *                             + MapOutputTracker::register_shuffle src/map_output_tracker.rs:168
 *   vb_shuffle_map_*       <- ShuffleDependencyTrait::do_shuffle_task  src/dependency.rs:96,164-229
 *                             (called from ShuffleMapTask::run, src/shuffle/shuffle_map_task.rs:86-90)
 *   vb_get_partition       <- HashPartitioner::get_partition      src/partitioner.rs:54-57 (+ hash :21-25)
 *   vb_shuffle_seal        <- register_map_outputs ("all map outputs registered")
 *                             src/scheduler/base_scheduler.rs:304-316
 *   vb_shuffle_reduce*     <- ShuffledRdd::compute                src/rdd/shuffled_rdd.rs:149-170
 *                             + ShuffleFetcher::fetch             src/shuffle/shuffle_fetcher.rs:16-119
 *   vb_join*               <- CoGroupedRdd::compute               src/rdd/co_grouped_rdd.rs:206-249
 *                             + PairRdd::join cross product       src/rdd/pair_rdd.rs:104-121
 *   vb_cogroup*            <- PairRdd::cogroup                    src/rdd/pair_rdd.rs:123-155
 *   vb_join_outer*         <- (absent from the reference: Spark's left/right/full outer joins)
 *   vb_shuffle_free        <- (the reference never evicts SHUFFLE_CACHE, src/env.rs:27)
 *   vb_slice               <- ParallelCollection::slice           src/rdd/parallel_collection_rdd.rs:116-145
 *   vb_shuffle_export_* / vb_shuffle_import
 *                          <- the shuffle data plane (hyper HTTP GET /shuffle/{sid}/{map}/{reduce},
 *                             src/shuffle/shuffle_manager.rs:176-251) when reduce partitions live on
 *                             other GPUs: rows packed by destination rank for one all-to-all-v.
 *
 * Conventions: plain pointers and sizes only.  Every call returns 0 (VB_OK) or a negative
 * vb_status; vb_last_error() gives a thread-local message.  No panics/exceptions cross the
 * boundary (the reference unwrap()s, dependency.rs:191-214).  Host pointers are caller-owned;
 * device memory is library-owned unless passed in as VB_DEVICE*.  Entry points may be called
 * concurrently from arbitrary OS threads (vega runs map tasks on a tokio blocking pool,
 * src/scheduler/local_scheduler.rs:336-352).  A context serialises the ENQUEUEING of its device work; a map
 * call with host input waits for its own completion with the context unlocked, its H2D copies run on a
 * separate copy stream through two staging halves, so concurrent map tasks keep PCIe and the SMs busy together.
 * Device work runs on the context's own stream (vb_ctx_stream): device buffers handed in must be complete
 * (producer stream synchronised) before the call; results are complete when a call returns.
 * There is NO CPU fallback: without a CUDA device every compute entry returns VB_ERR_CUDA.
 *
 * Rows are POD (K,V) with 64-bit K and V; `Aggregator` closures (src/aggregator.rs:8-16) are
 * replaced by named ops (vb_agg).  Arbitrary K/V/closures stay on vega's CPU path.
 */
#ifndef VEGA_B200_H
#define VEGA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VB_API __attribute__((visibility("default")))

typedef struct vb_ctx vb_ctx;   /* one CUDA device: streams, memory pool */
typedef struct vb_shuf vb_shuf; /* one shuffle_id: map outputs + sealed reduce-side results */

enum vb_status {
    VB_OK = 0,
    VB_ERR_INVALID = -1,     /* bad argument */
    VB_ERR_CUDA = -2,        /* CUDA runtime/driver error, or no device */
    VB_ERR_OOM = -3,         /* device or host allocation failed */
    VB_ERR_STATE = -4,       /* wrong phase (map after seal, reduce of a freed shuffle, ...) */
    VB_ERR_UNSUPPORTED = -5, /* dtype/agg combination not implemented */
    VB_ERR_TOO_LARGE = -6    /* more than 2^32-2 rows in one device-local shuffle / map partition */
};

enum vb_dtype { VB_U64 = 0, VB_I64 = 1, VB_F64 = 2 };

/* Aggregator (src/aggregator.rs).  GROUP = Default (Vec append, :33-52); SUM/MIN/MAX =
 * reduce_by_key(f) (src/rdd/pair_rdd.rs:65-80) for the named f; COUNT = count_by_value
 * (src/rdd/rdd.rs:450-459; values ignored, combiner is u64); COGROUP = the Vec-append
 * aggregator CoGroupedRdd installs per parent (src/rdd/co_grouped_rdd.rs:78-124), same
 * layout as GROUP; SORT = sort_by_key (absent from the reference, SURVEY.md F2).           */
enum vb_agg {
    VB_AGG_GROUP = 0,
    VB_AGG_SUM = 1,
    VB_AGG_MIN = 2,
    VB_AGG_MAX = 3,
    VB_AGG_COUNT = 4,
    VB_AGG_COGROUP = 5,
    VB_AGG_SORT = 6
};

/* VB_PART_HASH_METRO64: MetroHash64_1(key LE bytes, seed 0) % n_reduce (src/partitioner.rs:21-25,
 * 54-57; fasthash 0.4.0).  VB_PART_RANGE: contiguous key ranges (VB_AGG_SORT only).         */
enum vb_part { VB_PART_HASH_METRO64 = 0, VB_PART_RANGE = 1 };

/* where a caller buffer lives */
enum vb_loc {
    VB_HOST = 0,           /* host memory (pageable or pinned); copied inside the call */
    VB_DEVICE = 1,         /* device memory; consumed or copied before the call returns */
    VB_DEVICE_BORROWED = 2 /* device memory the caller keeps alive and unchanged until seal */
};

typedef struct vb_stats {
    uint64_t rows_in;          /* rows submitted through vb_shuffle_map_* */
    uint64_t rows_out;         /* result rows (distinct keys, or values for group ops) */
    uint64_t kernel_launches;  /* CUDA kernels this shuffle launched (ours, not memcpy/memset) */
    uint64_t h2d_bytes;        /* host→device bytes copied by the library */
    uint64_t d2h_bytes;        /* device→host bytes copied by the library */
    uint64_t table_slots;      /* largest hash-table capacity used */
    uint64_t table_restarts;   /* map tasks restarted with a larger table */
    double hot_kernel_ms;      /* summed device time of the dominant kernel (profiling on) */
    uint64_t hot_kernel_launches;
    uint64_t hot_kernel_rows;  /* rows those launches processed */
    double map_ms;             /* device time inside vb_shuffle_map_* (profiling on) */
    double seal_ms;            /* device time inside vb_shuffle_seal (profiling on) */
    uint64_t hot_kernel_variant; /* reduce ops: 1 = bulk-staged hash_agg (cp.async.bulk + mbarrier), 0 = register-staged */
} vb_stats;

/* ---- context ------------------------------------------------------------------------- */
VB_API int32_t vb_ctx_create(int32_t device_id, vb_ctx **out);
VB_API int32_t vb_ctx_destroy(vb_ctx *ctx);
VB_API int32_t vb_ctx_synchronize(vb_ctx *ctx);
/* profiling: bracket kernels with CUDA events on the launching stream (vb_stats *_ms) */
VB_API int32_t vb_ctx_set_profile(vb_ctx *ctx, int32_t on);
VB_API int32_t vb_ctx_device(vb_ctx *ctx);
/* the cudaStream_t all device work of this context is launched on (for event timing) */
VB_API void *vb_ctx_stream(vb_ctx *ctx);
/* bytes currently held by the context's (private) device memory pool / high-water mark */
VB_API int32_t vb_ctx_mem_info(vb_ctx *ctx, uint64_t *reserved, uint64_t *high_water);
/* give pool memory beyond keep_bytes back to the device (the pool otherwise keeps everything it ever used) */
VB_API int32_t vb_ctx_trim(vb_ctx *ctx, uint64_t keep_bytes);

/* ---- shuffle lifecycle ---------------------------------------------------------------- */
VB_API int32_t vb_shuffle_create(vb_ctx *ctx, uint64_t shuffle_id, uint32_t n_map, uint32_t n_reduce,
                                 int32_t key_dtype, int32_t val_dtype, int32_t agg, int32_t part,
                                 vb_shuf **out);
/* Hash the key as 4 LE bytes (Rust i32/u32 keys, widened to 64 bits by the caller) or 8. */
VB_API int32_t vb_shuffle_set_key_width(vb_shuf *s, uint32_t bytes);
/* Optional: expected number of distinct keys (sizes the first hash table; any value is safe). */
VB_API int32_t vb_shuffle_set_hint(vb_shuf *s, uint64_t expected_distinct);
/* One-process-per-GPU mode: this process is `rank` of `world`; reduce partition r is owned by
 * rank r % world.  Must precede the first map call.  world == 1 is the default.              */
VB_API int32_t vb_shuffle_set_dist(vb_shuf *s, uint32_t rank, uint32_t world);

/* do_shuffle_task for one map partition.  AoS = the reference's native Vec<(K,V)> layout
 * (16-byte rows); SoA = separate key/value arrays (vals may be NULL for VB_AGG_COUNT and
 * key-only VB_AGG_SORT).  Re-submitting a map_id overwrites it (stage resubmission,
 * src/scheduler/local_scheduler.rs:248-256).                                                */
VB_API int32_t vb_shuffle_map_aos(vb_shuf *s, uint32_t map_id, const void *rows, uint64_t n_rows, int32_t src_loc);
VB_API int32_t vb_shuffle_map_soa(vb_shuf *s, uint32_t map_id, const void *keys, const void *vals,
                                  uint64_t n_rows, int32_t src_loc);

/* world > 1 only.  export_prepare finishes the local map side and packs rows by destination
 * rank (combined rows for reduce ops, raw rows in map order for group ops); counts[world] gets
 * rows per destination.  export_buffers returns the packed device arrays (destination-major).
 * The host exchanges them (one all-to-all-v over NCCL) and hands the received rows, source-rank
 * major, to vb_shuffle_import (the buffers are borrowed until vb_shuffle_seal returns).  Then vb_shuffle_seal. */
VB_API int32_t vb_shuffle_export_prepare(vb_shuf *s, uint64_t *counts);
VB_API int32_t vb_shuffle_export_buffers(vb_shuf *s, void **keys_dev, void **vals_dev);
VB_API int32_t vb_shuffle_import(vb_shuf *s, const void *keys_dev, const void *vals_dev, const uint64_t *counts);

/* Fused exchange for GROUP/COGROUP shuffles (world > 1, one process per GPU on one NVLink/NVSwitch node):
 * the destination-rank partition kernel stores every row straight into the HBM of the rank that owns its
 * reduce partition (peer memory mapped with CUDA IPC), so there is no pack buffer and no separate
 * collective — the transfer overlaps the partitioning tile by tile.  Protocol (vega_b200/dist.py drives it):
 *   1. vb_shuffle_export_counts(s, counts[world])        rows this rank sends to each rank (histogram only)
 *   2. ranks all-gather the counts; each reserves its receive arena for sum_src counts[src][me] rows
 *      (16 B/row: keys[total] then vals[total]) with vb_ctx_arena_reserve -> 64-byte IPC handle + generation
 *   3. ranks all-gather the handles; vb_ctx_peer_open(ctx, peer, handle, generation, is_self) maps them (cached
 *      per generation; is_self != 0 for the caller's own rank)
 *   4. vb_shuffle_export_direct(s, dst_row_offset[world], dst_total_rows[world]) runs the scatter; it returns when
 *      this rank's stores are complete; the host then barriers all ranks
 *   5. vb_shuffle_import_arena(s, counts_from_each_src[world]); vb_shuffle_seal(s)
 * The arena is reused (and only grows) across shuffles of the context; a shuffle must be sealed before the
 * next one's export_direct targets the same arena.                                                            */
VB_API int32_t vb_ctx_arena_reserve(vb_ctx *ctx, uint64_t bytes, void *handle_out /*64 bytes*/, uint64_t *generation);
VB_API int32_t vb_ctx_peer_open(vb_ctx *ctx, uint32_t peer_rank, const void *handle /*64 bytes*/, uint64_t generation, int32_t is_self);
VB_API int32_t vb_shuffle_export_counts(vb_shuf *s, uint64_t *counts);
VB_API int32_t vb_shuffle_export_direct(vb_shuf *s, const uint64_t *dst_row_offset, const uint64_t *dst_total_rows);
VB_API int32_t vb_shuffle_import_arena(vb_shuf *s, const uint64_t *counts);

/* Free the arenas vb_ctx_arena_reserve outgrew.  Call after the barrier that follows the exchange: by then every
 * peer has re-opened this rank's current arena (vb_ctx_peer_open closes its mapping of the old one) — freeing an
 * exported allocation a peer still has mapped is undefined.                                                    */
VB_API int32_t vb_ctx_arena_release_retired(vb_ctx *ctx);

/* ---- the exchange itself, behind the C ABI (ShuffleFetcher::fetch, src/shuffle/shuffle_fetcher.rs:16-119;
 *      the tracker hand-shake it replaces: src/map_output_tracker.rs:168-265) ---------------------------------
 * One process per GPU.  vb_comm_unique_id (rank 0) produces the 128-byte NCCL unique id; the host bootstrap
 * (vega's tracker channel, torch.distributed, the TCP rendezvous in vega_b200/rendezvous.py, ...) hands it to every rank; vb_ctx_comm_init is
 * collective over the `world` ranks.  Then, per shuffle, instead of export_prepare / buffers / import:
 *
 *     vb_shuffle_map_*(...)  ...  vb_shuffle_exchange(s, VB_XCHG_AUTO);  vb_shuffle_seal(s);
 *
 * vb_shuffle_exchange is collective and runs entirely on the library's stream:
 *   VB_XCHG_NCCL  pack rows by destination rank (combined rows for reduce ops), all-gather the world x world
 *                 count matrix (one small collective + one D2H), then ONE ncclGroupStart .. ncclSend/ncclRecv
 *                 .. ncclGroupEnd carrying keys and values of every peer (a single all-to-all-v).
 *   VB_XCHG_P2P   GROUP/COGROUP: the fused exchange above — the partition kernel stores into the peers'
 *                 arenas; counts, arena sizes/generations ride one all-gather, IPC handles a second one only
 *                 when some arena had to grow; a stream-ordered all-gather is the closing barrier.
 *   VB_XCHG_AUTO  P2P for group ops, NCCL for reduce ops.
 * NCCL is dlopen'ed (libnccl.so.2) on first use.  vb_ctx_destroy / vb_ctx_comm_destroy are collective when a
 * communicator exists (peer mappings are closed before the arenas are freed).                                 */
#define VB_UNIQUE_ID_BYTES 128
enum vb_xchg { VB_XCHG_AUTO = 0, VB_XCHG_NCCL = 1, VB_XCHG_P2P = 2 };
typedef struct vb_xstats {
    uint64_t sent_rows;     /* rows that left this rank (excluding rows it keeps) */
    uint64_t recv_rows;
    uint64_t exchanges;
    double exchange_ms;     /* device time of the exchange (profiling on): NCCL group, or counts+scatter+barrier for P2P */
    int32_t kind;           /* vb_xchg actually used */
    int32_t pad;
    double prepare_wall_ms; /* host wall clock: finish the map side + pack by destination (merge, multisplit, their syncs) */
    double counts_wall_ms;  /* host wall clock: count all-gather + D2H */
    double post_wall_ms;    /* host wall clock: buffers + enqueueing the grouped send/recv (or handles + scatter + barrier) */
} vb_xstats;
VB_API int32_t vb_comm_unique_id(void *id_out /*VB_UNIQUE_ID_BYTES*/);
VB_API int32_t vb_ctx_comm_init(vb_ctx *ctx, const void *unique_id, uint32_t rank, uint32_t world);
VB_API int32_t vb_ctx_comm_destroy(vb_ctx *ctx);
VB_API int32_t vb_ctx_comm_info(vb_ctx *ctx, uint32_t *rank, uint32_t *world, int32_t *nccl_version);
VB_API int32_t vb_shuffle_exchange(vb_shuf *s, int32_t mode);
VB_API int32_t vb_shuffle_exchange_stats(vb_shuf *s, vb_xstats *out);

/* All map outputs are registered: run the reduce side for every partition this rank owns.
 * world == 1: every map_id in [0, n_map) must have been submitted.                          */
VB_API int32_t vb_shuffle_seal(vb_shuf *s);
VB_API int32_t vb_shuffle_is_sealed(vb_shuf *s);

/* ShuffledRdd::compute for one reduce partition.  Both calls BLOCK until the shuffle is sealed
 * (the reference polls the map-output tracker, src/map_output_tracker.rs:122-132,220-231).
 *   reduce ops : out_keys[n_keys], out_combined[n_keys]            (n_vals == 0)
 *   group ops  : out_keys[n_keys], out_offsets[n_keys+1], out_vals[n_vals]  (CSR; each key's
 *                values in input order: map-id order, then encounter order — tests/test_pair_rdd.rs:30-36)
 *   sort       : out_keys[n_keys] ascending, out_combined[n_keys] = payload (if any)
 * Key order within a partition is unspecified (the reference's is HashMap order).
 * NULL output pointers are skipped.  dst_loc: VB_HOST or VB_DEVICE.                          */
VB_API int32_t vb_shuffle_reduce_size(vb_shuf *s, uint32_t reduce_id, uint64_t *n_keys, uint64_t *n_vals);
VB_API int32_t vb_shuffle_reduce(vb_shuf *s, uint32_t reduce_id, void *out_keys, void *out_combined,
                                 uint64_t *out_offsets, void *out_vals, int32_t dst_loc);

/* Inner join of two sealed GROUP/COGROUP shuffles with equal n_reduce, for one partition:
 * per key `for v in left { for w in right }` (src/rdd/pair_rdd.rs:109-115).                  */
VB_API int32_t vb_join_size(vb_shuf *left, vb_shuf *right, uint32_t reduce_id, uint64_t *n_out);
VB_API int32_t vb_join(vb_shuf *left, vb_shuf *right, uint32_t reduce_id, void *out_k, void *out_v, void *out_w,
                       int32_t dst_loc);

/* PairRdd::cogroup (src/rdd/pair_rdd.rs:123-155, co_grouped_rdd.rs:206-249) for reduce partition r
 * of two sealed GROUP/COGROUP shuffles with the same n_reduce and key width.  Keys in union order:
 * the left side's keys in its CSR order, then the right-only keys in the right CSR order.  Each
 * key's values per side in input order; a key absent on a side has an empty list there.
 * Argument checks, blocking and error codes as vb_join; 0 keys on a rank that does not own r.    */
VB_API int32_t vb_cogroup_size(vb_shuf *left, vb_shuf *right, uint32_t reduce_id,
                               uint64_t *n_keys, uint64_t *n_left_vals, uint64_t *n_right_vals);
VB_API int32_t vb_cogroup(vb_shuf *left, vb_shuf *right, uint32_t reduce_id,
                          void *out_keys,        /* n_keys */
                          uint64_t *out_offs_l,  /* n_keys + 1, partition-local, [0] = 0 */
                          void *out_vals_l,      /* n_left_vals */
                          uint64_t *out_offs_r,  /* n_keys + 1 */
                          void *out_vals_r,      /* n_right_vals */
                          int32_t dst_loc);      /* VB_HOST | VB_DEVICE, as vb_join */

/* Left / right / full outer join: absent from the reference; Spark semantics; parity unpinned.
 * Rows of one key are contiguous, keys in the cogroup's union order.  A key with values on both
 * sides gives `for v in vs { for w in ws }` (as vb_join); LEFT_OUTER adds (v, absent) for a
 * left-only key, RIGHT_OUTER (absent, w) for a right-only key, FULL_OUTER both.  An absent value
 * is written as 0 and its bit is clear in out_valid[i] (VB_JOIN_HAS_V | VB_JOIN_HAS_W on matched
 * rows).  A bad kind is VB_ERR_INVALID; otherwise checks, blocking and codes as vb_join.        */
enum vb_join_kind { VB_JOIN_LEFT_OUTER = 1, VB_JOIN_RIGHT_OUTER = 2, VB_JOIN_FULL_OUTER = 3 };
enum vb_join_valid { VB_JOIN_HAS_V = 1, VB_JOIN_HAS_W = 2 };   /* bits of out_valid[i] */
VB_API int32_t vb_join_outer_size(vb_shuf *left, vb_shuf *right, uint32_t reduce_id, int32_t kind, uint64_t *n_out);
VB_API int32_t vb_join_outer(vb_shuf *left, vb_shuf *right, uint32_t reduce_id, int32_t kind,
                             void *out_k, void *out_v, void *out_w, uint8_t *out_valid /* may be NULL */,
                             int32_t dst_loc);

/* ---- SURVEY §8(f) N1: bincode blobs — the payload format of SHUFFLE_CACHE ------------------------
 * The reference serialises every (map, reduce) bucket with bincode 1.2.1 defaults (src/dependency.rs:213-214:
 * little-endian, fixed-width integers, u64 length prefixes) and decodes it in the fetcher
 * (src/shuffle/shuffle_fetcher.rs:85).  These entry points speak that format so GPU results can be
 * served to, and CPU-produced buckets consumed from, unmodified vega executors:
 *   Vec<(u64,u64)>      = u64 n | n x (u64 k, u64 c)                       (reduce ops, sort)
 *   Vec<(u64,Vec<u64>)> = u64 n | n x (u64 k, u64 len, len x u64)          (group ops)
 * vb_shuffle_reduce_blob encodes one sealed reduce partition; vb_shuffle_map_blob submits one
 * map-side-COMBINED bucket as the output of map task `map_id` (combiners are merged with
 * merge_combiners, so partial counts are summed).  A blob whose length field disagrees with its
 * size is rejected with VB_ERR_INVALID (the reference's DeserializationError).                   */
VB_API int32_t vb_shuffle_reduce_blob_size(vb_shuf *s, uint32_t reduce_id, uint64_t *n_bytes);
VB_API int32_t vb_shuffle_reduce_blob(vb_shuf *s, uint32_t reduce_id, void *out_blob, int32_t dst_loc);
VB_API int32_t vb_shuffle_map_blob(vb_shuf *s, uint32_t map_id, const void *blob, uint64_t n_bytes, int32_t src_loc);

VB_API int32_t vb_shuffle_free(vb_shuf *s);
VB_API int32_t vb_shuffle_stats(vb_shuf *s, vb_stats *out);
VB_API const char *vb_last_error(void);

/* ---- host-side pieces of the path ------------------------------------------------------ */
/* MetroHash64_1 of the key's 4 or 8 LE bytes, seed 0 (src/partitioner.rs:21-25). */
VB_API uint64_t vb_hash_key(uint64_t key, uint32_t key_width);
/* HashPartitioner::get_partition (src/partitioner.rs:54-57). */
VB_API uint32_t vb_get_partition(uint64_t key, uint32_t key_width, uint32_t n_reduce);
/* ParallelCollection::slice: writes slice starts (and n as the last entry) into
 * starts[min(n,num_slices)+2] and returns the number of slices (n+1 when n < num_slices).  */
VB_API uint64_t vb_slice(uint64_t n, uint64_t num_slices, uint64_t *starts);

/* Context::range (src/context.rs:419-431): the u64 sequence (start..=end).step_by(step) as a device-resident
 * source — SURVEY §8(f) N3: no host array, no H2D.  vb_range_len = number of elements; out_dev holds that many. */
VB_API uint64_t vb_range_len(uint64_t start, uint64_t end, uint64_t step);
VB_API int32_t vb_range(vb_ctx *ctx, void *out_dev, uint64_t start, uint64_t end, uint64_t step);

/* ---- synthetic input, generated on the device (bench / parity tests) -------------------- */
/* Row i (i = first .. first+n-1):
 *   VB_GEN_UNIFORM  rank = splitmix64(seed_k+i) % n_distinct
 *   VB_GEN_ZIPF     rank = Zipf(zipf_s) over [0,n_distinct) by inverse CDF, u = splitmix64(seed_k+i)/2^64
 *   VB_GEN_UNIQUE   rank = rank_base + i   (each rank exactly once: join inputs)
 * key = splitmix64(rank ^ 0xA5A5A5A5A5A5A5A5) (a bijection: distinct ranks give distinct keys);
 * val = splitmix64(seed_v+i) & 0xFFFFF.  Writes AoS rows (rows_dev) if non-NULL, else SoA
 * keys_dev / vals_dev (vals_dev may be NULL).  Same stream as oracle/vega_oracle.c:vo_gen_uniform. */
enum vb_gen { VB_GEN_UNIFORM = 0, VB_GEN_ZIPF = 1, VB_GEN_UNIQUE = 2 };
VB_API int32_t vb_gen_pairs(vb_ctx *ctx, void *rows_dev, void *keys_dev, void *vals_dev, uint64_t first, uint64_t n,
                            int32_t mode, uint64_t n_distinct, uint64_t rank_base, uint64_t seed_k, uint64_t seed_v,
                            double zipf_s);

/* Device time and launch count per kernel class (profiling on): 0 hash_agg (map-side combine),
 * 1 dict build, 2 merge, 3 rp_hist, 4 rp_scan, 5 rp_scatter, 6 misc, 7 join.                   */
VB_API int32_t vb_shuffle_kernel_time(vb_shuf *s, int32_t klass, double *ms, uint64_t *launches);

/* library build info: "vega_b200 <version> sm_100a" */
VB_API const char *vb_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VEGA_B200_H */
