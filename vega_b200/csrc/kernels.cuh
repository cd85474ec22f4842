// kernels.cuh — hand-written sm_100a kernels of the shuffle + aggregation path.
//
//   hash_agg_kernel   map-side combine (dependency.rs:191-210) and reduce-side merge
//                     (shuffled_rdd.rs:154-164) as one streaming pass into an L2-resident
//                     open-addressing table: 128-bit evict-first loads, one probe + one RED per row.
//                     OPK_DICT variant builds the key dictionary for group_by_key / cogroup.
//   rp_hist / rp_scatter   one stable radix pass (multisplit by hash(K) % nparts, LSD sort digits):
//                     warp match-any ranking, shared-memory staged tiles, coalesced run writes.
//   scan kernels, CSR boundary, join probe/expand, generators.
//
// Integer / indexing work: HBM- and L2-bound, no tensor cores by design.
#pragma once
#include "common.cuh"

namespace vb {

// ---------------------------------------------------------------------------------------------
// Hash table: open addressing over 4-key buckets, keys and accumulators in separate arrays.
//
// Measured on B200 (profiles/r1_micro_*.log): a random 8..32-byte read of an L2-resident table
// sustains ~2.5e11 probes/s and a 64-bit RED ~1.5e11/s, but a *dependent* linear-probing loop
// (30-46 % of rows need a second probe at load 0.48) serialises L2 latencies inside divergent
// warps and ran 6x slower.  So a bucket is the 4 keys of one 32-byte sector, fetched with a single
// 256-bit load (LDG.E.NA.256): at load <= 0.6 almost every row resolves in its first probe and the
// kernel issues all probes of a tile before consuming any.  L1::no_allocate on the probes keeps
// the REDs that follow from invalidating L1 lines.
// ---------------------------------------------------------------------------------------------
struct Table {
    u64 *keys;    // [cap + 4]: keys[cap] is the marker of the special slot (1 = EMPTY_KEY present)
    u64 *accs;    // [cap + 4]: combiner per slot (reduce ops); unused by the dictionary
    u32 log_cap;  // cap = 1 << log_cap slots = cap / 4 buckets; log_cap >= 2
};
constexpr u64 EMPTY_KEY = ~0ull;
constexpr u32 BUCKET = 4;
VB_HD size_t table_bytes(u32 log_cap) { return (((size_t)1 << log_cap) + BUCKET) * 16; }
VB_HD Table table_at(void *base, u32 log_cap)
{
    Table t;
    t.keys = (u64 *)base;
    t.accs = (u64 *)base + (((size_t)1 << log_cap) + BUCKET);
    t.log_cap = log_cap;
    return t;
}

struct TableCtl {
    u32 abort;        // set by the kernel: table too full / probe sequence too long → host restarts
    u32 pad;
    unsigned long long n_inserted;
};

enum : int { IN_AOS = 0, IN_SOA = 1, IN_TABLE = 2 };
enum : int { OPK_ADD_U64 = 0, OPK_ADD_F64 = 1, OPK_MIN_U64 = 2, OPK_MAX_U64 = 3, OPK_COUNT = 4, OPK_DICT = 5 };

VB_HD u64 op_identity(int opk) { return opk == OPK_MIN_U64 ? ~0ull : 0ull; }

// Table accesses can carry an L2 evict_last hint (the stream is evict_first): A/B-measured, see VB_TABLE_EVICT_LAST.
#ifndef VB_TABLE_EVICT_LAST
#define VB_TABLE_EVICT_LAST 0
#endif
VB_D u64 table_policy()
{
#if VB_TABLE_EVICT_LAST
    return policy_evict_last();
#else
    return 0;
#endif
}

template <int OPK>
VB_D void op_red_hint(u64 *acc, u64 v, u64 pol)
{
#if VB_TABLE_EVICT_LAST
    if (OPK == OPK_ADD_U64) asm volatile("red.global.add.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(acc), "l"(v), "l"(pol) : "memory");
    else if (OPK == OPK_COUNT) asm volatile("red.global.add.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(acc), "l"(1ull), "l"(pol) : "memory");
    else if (OPK == OPK_ADD_F64) asm volatile("red.global.add.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(acc), "d"(__longlong_as_double((long long)v)), "l"(pol) : "memory");
    else if (OPK == OPK_MIN_U64) asm volatile("red.global.min.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(acc), "l"(v), "l"(pol) : "memory");
    else if (OPK == OPK_MAX_U64) asm volatile("red.global.max.L2::cache_hint.u64 [%0], %1, %2;" ::"l"(acc), "l"(v), "l"(pol) : "memory");
#else
    (void)pol;
    if (OPK == OPK_ADD_U64) atomicAdd((unsigned long long *)acc, (unsigned long long)v);
    else if (OPK == OPK_COUNT) atomicAdd((unsigned long long *)acc, 1ull);
    else if (OPK == OPK_ADD_F64) atomicAdd((double *)acc, __longlong_as_double((long long)v));
    else if (OPK == OPK_MIN_U64) atomicMin((unsigned long long *)acc, (unsigned long long)v);
    else if (OPK == OPK_MAX_U64) atomicMax((unsigned long long *)acc, (unsigned long long)v);
#endif
}

template <int OPK>
VB_D void op_red(u64 *acc, u64 v)
{
    if (OPK == OPK_ADD_U64) atomicAdd((unsigned long long *)acc, (unsigned long long)v);
    else if (OPK == OPK_COUNT) atomicAdd((unsigned long long *)acc, 1ull);
    else if (OPK == OPK_ADD_F64) atomicAdd((double *)acc, __longlong_as_double((long long)v));
    else if (OPK == OPK_MIN_U64) atomicMin((unsigned long long *)acc, (unsigned long long)v);
    else if (OPK == OPK_MAX_U64) atomicMax((unsigned long long *)acc, (unsigned long long)v);
}

__global__ void table_init_kernel(Table t, u64 identity)
{
    const u64 cap = 1ull << t.log_cap;
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (; i < cap + BUCKET; i += stride) {
        t.keys[i] = (i >= cap) ? 0ull : EMPTY_KEY;
        t.accs[i] = identity;
    }
}

struct Bucket4 { u64 k0, k1, k2, k3; };

// one 32-byte sector: 4 candidate keys
VB_D Bucket4 ld_bucket(const u64 *p)
{
    Bucket4 b;
    asm volatile("ld.global.L1::no_allocate.v4.u64 {%0, %1, %2, %3}, [%4];"
                 : "=l"(b.k0), "=l"(b.k1), "=l"(b.k2), "=l"(b.k3)
                 : "l"(p));
    return b;
}
VB_D Bucket4 ld_bucket_hint(const u64 *p, u64 pol)
{
#if VB_TABLE_EVICT_LAST
    Bucket4 b;
    asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.u64 {%0, %1, %2, %3}, [%4], %5;"
                 : "=l"(b.k0), "=l"(b.k1), "=l"(b.k2), "=l"(b.k3)
                 : "l"(p), "l"(pol));
    return b;
#else
    (void)pol;
    return ld_bucket(p);
#endif
}
VB_D int bucket_find(const Bucket4 &b, u64 key)
{
    return b.k0 == key ? 0 : b.k1 == key ? 1 : b.k2 == key ? 2 : b.k3 == key ? 3 : -1;
}

constexpr int HA_THREADS = 256;
constexpr int HA_ROWS = 4;
constexpr int HA_TILE = HA_THREADS * HA_ROWS;
constexpr u32 HA_MAX_PROBE = 256;   // buckets

VB_D u64 home_bucket(u64 key, u32 log_cap) { return slot_hash(key) >> (64 - (log_cap - 2)); }

// Resolve `key` starting from bucket `b` whose content `bk` is already loaded: find it, or claim the
// first empty slot with a CAS, or move on to the next bucket.  Slots only ever go EMPTY → key and are
// claimed first-empty-first, so a key can never end up in two slots (a stale view is an older view).
template <int OPK>
VB_D bool table_resolve(const Table &t, u64 b, Bucket4 bk, u64 key, u64 v, u32 &slot_idx, u32 &inserted)
{
    const u64 nb_mask = (1ull << (t.log_cap - 2)) - 1;
#pragma unroll 1
    for (u32 probe = 0; probe < HA_MAX_PROBE; ++probe) {
        int hit = bucket_find(bk, key);
        if (hit < 0) {
            const int e = bucket_find(bk, EMPTY_KEY);
            if (e < 0) {
                b = (b + 1) & nb_mask;
            } else {
                const u64 old = atomicCAS((unsigned long long *)&t.keys[4 * b + e], (unsigned long long)EMPTY_KEY, (unsigned long long)key);
                if (old == EMPTY_KEY) { ++inserted; hit = e; }
                else if (old == key) hit = e;
            }
        }
        if (hit >= 0) {
            const u64 s = 4 * b + (u64)hit;
            op_red<OPK>(&t.accs[s], v);
            slot_idx = (u32)s;
            return true;
        }
        bk = ld_bucket(&t.keys[4 * b]);
    }
    return false;
}

// ---- per-CTA hot-key cache (skewed keys) -------------------------------------------------------
// With Zipf(1.1) keys the hottest key owns 12 % of the rows: 1.2e8 REDs to ONE L2 address serialise
// (measured 104 ms per 1e9 rows vs 10 ms uniform).  Each CTA therefore keeps a small 2-choice cache
// of (key, partial combiner) in shared memory: rows whose key is cached are combined with a
// shared-memory atomic and never reach L2; the cache is flushed into the table once, at CTA exit.
// Keys are cached first-come (hot keys come first with high probability).  For uniformly distributed
// keys nothing hits, so every CTA measures its hit rate over its first 16 tiles and switches the
// cache off below 1/16.
constexpr int HC_SLOTS = 1024;
#ifndef VB_HC_ENABLE
#define VB_HC_ENABLE 1
#endif

template <int OPK>
VB_D void op_shared(u64 *acc, u64 v)
{
    if (OPK == OPK_ADD_U64) atomicAdd((unsigned long long *)acc, (unsigned long long)v);
    else if (OPK == OPK_COUNT) atomicAdd((unsigned long long *)acc, 1ull);
    else if (OPK == OPK_ADD_F64) atomicAdd((double *)acc, __longlong_as_double((long long)v));
    else if (OPK == OPK_MIN_U64) atomicMin((unsigned long long *)acc, (unsigned long long)v);
    else if (OPK == OPK_MAX_U64) atomicMax((unsigned long long *)acc, (unsigned long long)v);
}

// 0: not absorbed (row goes to the table); 1: hit an already cached key; 2: claimed an empty cache slot
template <int OPK>
VB_D int cache_combine(u64 *hc_keys, u64 *hc_acc, u64 h, u64 key, u64 v)
{
    const u32 i1 = (u32)h & (HC_SLOTS - 1), i2 = (u32)(h >> 10) & (HC_SLOTS - 1);
    const u64 c1 = hc_keys[i1];
    if (c1 == key) { op_shared<OPK>(&hc_acc[i1], v); return 1; }
    const u64 c2 = hc_keys[i2];
    if (c2 == key) { op_shared<OPK>(&hc_acc[i2], v); return 1; }
    u32 slot;
    if (c1 == EMPTY_KEY) slot = i1;
    else if (c2 == EMPTY_KEY) slot = i2;
    else return 0;
    const u64 old = atomicCAS((unsigned long long *)&hc_keys[slot], (unsigned long long)EMPTY_KEY, (unsigned long long)key);
    if (old == EMPTY_KEY) { op_shared<OPK>(&hc_acc[slot], v); return 2; }
    if (old == key) { op_shared<OPK>(&hc_acc[slot], v); return 1; }
    return 0;
}

// The per-tile work shared by the register-staged and the bulk-staged kernels: thread-private rows
// k/v/ok (HA_ROWS of them, row j of the thread is input row row0 + j * HA_THREADS) → special key,
// hot-key cache, then lockstep probe rounds with one RED per resolved row.
template <int OPK, int TX, bool CACHE, int ROWS>
VB_D void ha_process_rows(const Table &t, TableCtl *ctl, u64 (&k)[ROWS], u64 (&v)[ROWS], bool (&ok)[ROWS], u64 row0,
                          u32 *__restrict__ slot_out, u64 *hc_keys, u64 *hc_acc, bool use_cache, u32 &my_inserts, u32 &my_hits)
{
    const u64 cap = 1ull << t.log_cap;
    const u64 tpol = table_policy();
    const u32 hshift = 64 - (t.log_cap - 2);
    u64 h[ROWS];
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
        h[j] = slot_hash(k[j]);
        if (TX != TX_NONE) v[j] = tx_fwd(v[j], TX);
        if (ok[j] && k[j] == EMPTY_KEY) {           // a real key equal to the empty marker: special slot
            t.keys[cap] = 1ull;
            op_red<OPK>(&t.accs[cap], v[j]);
            if (OPK == OPK_DICT) st_stream_u32(slot_out + row0 + (u64)j * HA_THREADS, (u32)cap);
            ok[j] = false;
        }
    }
    if (CACHE && use_cache) {
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
            if (!ok[j]) continue;
            const int c = cache_combine<OPK>(hc_keys, hc_acc, h[j], k[j], v[j]);
            if (c) { ok[j] = false; my_hits += (c == 1); }
        }
    }
    // Probe rounds run in lockstep over the ROWS rows of a thread: every round first consumes the
    // buckets loaded by the previous one, then issues the next probes of all unresolved rows together,
    // so a tile costs max-over-rows (not sum-over-rows) dependent L2 latencies.
    Bucket4 bk[ROWS];
    u64 bidx[ROWS];
    const u64 nb_mask = (1ull << (t.log_cap - 2)) - 1;
#pragma unroll
    for (int j = 0; j < ROWS; ++j) {
        bidx[j] = h[j] >> hshift;
        if (ok[j]) bk[j] = ld_bucket_hint(&t.keys[4 * bidx[j]], tpol);
    }
    bool pending = true;
#pragma unroll 1
    for (u32 probe = 0; pending && probe < HA_MAX_PROBE; ++probe) {
        pending = false;
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
            if (!ok[j]) continue;
            int hit = bucket_find(bk[j], k[j]);
            if (hit < 0) {
                const int e = bucket_find(bk[j], EMPTY_KEY);
                if (e < 0) {
                    bidx[j] = (bidx[j] + 1) & nb_mask;                    // bucket full: next bucket
                } else {
                    const u64 old = atomicCAS((unsigned long long *)&t.keys[4 * bidx[j] + e], (unsigned long long)EMPTY_KEY,
                                              (unsigned long long)k[j]);
                    if (old == EMPTY_KEY) { ++my_inserts; hit = e; }
                    else if (old == k[j]) hit = e;                        // else: lost the slot, re-read this bucket
                }
            }
            if (hit >= 0) {
                const u64 sl = 4 * bidx[j] + (u64)hit;
                op_red_hint<OPK>(&t.accs[sl], v[j], tpol);
                if (OPK == OPK_DICT) st_stream_u32(slot_out + row0 + (u64)j * HA_THREADS, (u32)sl);
                ok[j] = false;
            } else {
                pending = true;
            }
        }
        if (pending) {
#pragma unroll
            for (int j = 0; j < ROWS; ++j)
                if (ok[j]) bk[j] = ld_bucket_hint(&t.keys[4 * bidx[j]], tpol);
        }
    }
    if (pending) atomicExch(&ctl->abort, 1u);   // probe chain longer than HA_MAX_PROBE buckets
}

// One pass over n rows.  IN_AOS: a = rows (16 B each).  IN_SOA: a = keys, b = vals (b may be
// NULL for COUNT/DICT).  IN_TABLE: a/b = keys/accs of a source table of n-1 slots + the special slot.
// TX: order-preserving value transform applied on load (MIN/MAX over i64/f64).
template <int IN, int OPK, int TX>
__global__ void __launch_bounds__(HA_THREADS, 3)   // 3 CTAs/SM measured best (profiles/r1_micro_v4_bucketized.log)
hash_agg_kernel(const u64 *__restrict__ a, const u64 *__restrict__ b, u64 n, Table t, TableCtl *ctl, u64 max_inserts,
                u32 *__restrict__ slot_out)
{
    constexpr bool CACHE = VB_HC_ENABLE && (OPK != OPK_DICT) && (IN != IN_TABLE);
    constexpr int OPK_FLUSH = (OPK == OPK_COUNT) ? OPK_ADD_U64 : OPK;      // partial counts are summed
    __shared__ u32 s_inserts;
    __shared__ u32 s_abort;
    __shared__ u32 s_hits;
    __shared__ u64 hc_keys[CACHE ? HC_SLOTS : 1];
    __shared__ u64 hc_acc[CACHE ? HC_SLOTS : 1];
    const u32 tid = threadIdx.x;
    if (tid == 0) { s_inserts = 0; s_abort = 0; s_hits = 0; }
    if (CACHE)
        for (u32 i = tid; i < HC_SLOTS; i += HA_THREADS) { hc_keys[i] = EMPTY_KEY; hc_acc[i] = op_identity(OPK); }
    __syncthreads();
    const u64 pol = policy_evict_first();
    const u64 n_tiles = (n + HA_TILE - 1) / HA_TILE;
    u32 my_inserts = 0, my_hits = 0;
    u32 iter = 0;
    bool use_cache = CACHE;
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++iter) {
        const u64 base = tile * HA_TILE;
        u64 k[HA_ROWS], v[HA_ROWS];
        bool ok[HA_ROWS];
#pragma unroll
        for (int j = 0; j < HA_ROWS; ++j) {
            const u64 idx = base + (u64)j * HA_THREADS + tid;
            ok[j] = idx < n;
            k[j] = 0; v[j] = 0;
            if (ok[j]) {
                if (IN == IN_AOS) {
                    ulonglong2 r = ld_stream_u64x2(a + 2 * idx, pol);
                    k[j] = r.x; v[j] = r.y;
                } else if (IN == IN_SOA) {
                    k[j] = ld_stream_u64(a + idx, pol);
                    if (OPK != OPK_COUNT && OPK != OPK_DICT) v[j] = ld_stream_u64(b + idx, pol);
                } else {
                    k[j] = ld_stream_u64(a + idx, pol);
                    v[j] = ld_stream_u64(b + idx, pol);
                    if (idx == n - 1) { ok[j] = (k[j] == 1ull); k[j] = EMPTY_KEY; }   // special slot
                    else if (k[j] == EMPTY_KEY) ok[j] = false;                       // unoccupied
                }
            }
        }
        ha_process_rows<OPK, TX, CACHE, HA_ROWS>(t, ctl, k, v, ok, base + tid, slot_out, hc_keys, hc_acc, use_cache, my_inserts, my_hits);
        if ((iter & 15u) == 15u) {   // periodic load-factor check (+ cache verdict); iter is CTA-uniform
            u32 w = __reduce_add_sync(0xffffffffu, my_inserts);
            my_inserts = 0;
            if ((tid & 31u) == 0 && w) atomicAdd(&s_inserts, w);
            if (CACHE && iter == 15u) {
                u32 hw = __reduce_add_sync(0xffffffffu, my_hits);
                if ((tid & 31u) == 0 && hw) atomicAdd(&s_hits, hw);
            }
            __syncthreads();
            if (tid == 0) {
                u32 c = s_inserts;
                s_inserts = 0;
                u64 tot = atomicAdd(&ctl->n_inserted, (unsigned long long)c) + c;
                u32 ab = ld_volatile_u32(&ctl->abort);
                if (tot > max_inserts) { ab = 1; atomicExch(&ctl->abort, 1u); }
                s_abort = ab;
            }
            __syncthreads();
            if (s_abort) return;
            if (CACHE && iter == 15u && s_hits * 16u < 16u * HA_TILE) use_cache = false;   // < 1/16 of the first 16 tiles
        }
    }
    if (CACHE) {   // flush the cache into the table (merge op)
        __syncthreads();
        for (u32 i = tid; i < HC_SLOTS; i += HA_THREADS) {
            const u64 key = hc_keys[i];
            if (key == EMPTY_KEY) continue;
            const u64 hb = home_bucket(key, t.log_cap);
            u32 slot = 0;
            if (!table_resolve<OPK_FLUSH>(t, hb, ld_bucket(&t.keys[4 * hb]), key, hc_acc[i], slot, my_inserts)) atomicExch(&ctl->abort, 1u);
        }
    }
    u32 w = __reduce_add_sync(0xffffffffu, my_inserts);
    if ((tid & 31u) == 0 && w) atomicAdd(&s_inserts, w);
    __syncthreads();
    if (tid == 0 && s_inserts) atomicAdd(&ctl->n_inserted, (unsigned long long)s_inserts);
}

// ---- bulk-staged variant (TMA engine) ---------------------------------------------------------------
// Same aggregation, different input path.  ncu on the register-staged kernel above shows the SM's
// L1TEX→XBAR request port as the busiest unit (l1tex__m_l1tex2xbar_req_cycles_active 81 %; one request
// per cycle per SM, and a random probe, a RED and every 128 B of the stream each cost one), with the
// port idle whenever all resident CTAs sit in the DRAM-latency phase of their tile.  Here a producer
// warp keeps HB_STAGES input tiles in flight per CTA with cp.async.bulk + mbarrier (no registers, no
// LSU instructions for the stream); the 8 consumer warps only ever wait on L2-latency probes, so the
// request port stays busy.  Full tiles only (16-byte aligned, 16 KB each); the host sends inputs with
// unaligned bases to the register-staged kernel, and the sub-tile tail is read with plain loads.
#ifndef VB_HB_STAGES
#define VB_HB_STAGES 3
#endif
// 2 rows per thread x 4 CTAs per SM measured best on B200 (profiles/r2_micro_request_roof.log: 2.14 ms per 2.5e8 rows
// vs 2.51 for 4 x 3, 2.19 for 4 x 2(4 stages), 2.17 for the register-staged kernel)
#ifndef VB_HB_ROWS
#define VB_HB_ROWS 2
#endif
#ifndef VB_HB_CTAS
#define VB_HB_CTAS 4
#endif
constexpr int HB_STAGES = VB_HB_STAGES;
constexpr int HB_ROWS = VB_HB_ROWS;             // rows per consumer thread per tile
constexpr int HB_TILE = HA_THREADS * HB_ROWS;
constexpr int HB_THREADS = HA_THREADS + 32;     // 8 consumer warps + 1 producer warp
constexpr size_t hb_smem_bytes(bool has_vals) { return (size_t)HB_STAGES * HB_TILE * (has_vals ? 16 : 8); }

template <int IN, int OPK, int TX>
__global__ void __launch_bounds__(HB_THREADS, VB_HB_CTAS)
hash_agg_bulk_kernel(const u64 *__restrict__ a, const u64 *__restrict__ b, u64 n, Table t, TableCtl *ctl, u64 max_inserts,
                     u32 *__restrict__ slot_out)
{
    static_assert(IN == IN_AOS || IN == IN_SOA, "table merges use hash_agg_kernel");
    constexpr bool CACHE = VB_HC_ENABLE && (OPK != OPK_DICT);
    constexpr int OPK_FLUSH = (OPK == OPK_COUNT) ? OPK_ADD_U64 : OPK;
    constexpr bool HAS_V = (IN == IN_AOS) || (OPK != OPK_COUNT && OPK != OPK_DICT);
    constexpr u32 STAGE_BYTES = HB_TILE * (HAS_V ? 16 : 8);
    extern __shared__ __align__(128) unsigned char hb_stage[];      // [HB_STAGES][STAGE_BYTES]
    __shared__ __align__(8) u64 full_bar[HB_STAGES];
    __shared__ __align__(8) u64 empty_bar[HB_STAGES];
    __shared__ u32 s_inserts;
    __shared__ u32 s_abort;
    __shared__ u32 s_hits;
    __shared__ u64 hc_keys[CACHE ? HC_SLOTS : 1];
    __shared__ u64 hc_acc[CACHE ? HC_SLOTS : 1];
    const u32 tid = threadIdx.x;
    if (tid == 0) {
        s_inserts = 0; s_abort = 0; s_hits = 0;
#pragma unroll
        for (int s = 0; s < HB_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], HA_THREADS / 32); }
        mbar_fence_init();
    }
    if (CACHE)
        for (u32 i = tid; i < HC_SLOTS; i += HB_THREADS) { hc_keys[i] = EMPTY_KEY; hc_acc[i] = op_identity(OPK); }
    __syncthreads();
    const u64 n_full = n / HB_TILE;                         // tiles that go through the copy engine

    if (tid >= HA_THREADS) {                                // ===== producer warp =====
        if (tid == HA_THREADS) {
            const u64 pol = policy_evict_first();
            u32 i = 0;
            for (u64 tile = blockIdx.x; tile < n_full; tile += gridDim.x, ++i) {
                const u32 s = i % HB_STAGES;
                if (i >= HB_STAGES) mbar_wait(&empty_bar[s], ((i / HB_STAGES) & 1u) ^ 1u);   // consumers released the slot
                unsigned char *dst = hb_stage + (size_t)s * STAGE_BYTES;
                mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                if (IN == IN_AOS) {
                    bulk_g2s(dst, a + 2 * tile * HB_TILE, STAGE_BYTES, &full_bar[s], pol);
                } else {
                    bulk_g2s(dst, a + tile * HB_TILE, HB_TILE * 8, &full_bar[s], pol);
                    if (HAS_V) bulk_g2s(dst + HB_TILE * 8, b + tile * HB_TILE, HB_TILE * 8, &full_bar[s], pol);
                }
            }
        }
        return;                                             // every copy it issued is awaited by the consumers below
    }

    // ===== consumer warps =====
    u32 my_inserts = 0, my_hits = 0;
    u32 iter = 0;
    bool use_cache = CACHE;
    bool drain = false;        // after an abort: keep the pipeline moving (copies in flight target this CTA's smem), skip the work
    for (u64 tile = blockIdx.x; tile < n_full; tile += gridDim.x, ++iter) {
        const u32 s = iter % HB_STAGES;
        mbar_wait(&full_bar[s], (iter / HB_STAGES) & 1u);
        const unsigned char *src = hb_stage + (size_t)s * STAGE_BYTES;
        u64 k[HB_ROWS], v[HB_ROWS];
        bool ok[HB_ROWS];
#pragma unroll
        for (int j = 0; j < HB_ROWS; ++j) {
            const u32 r = (u32)j * HA_THREADS + tid;
            ok[j] = !drain;
            if (IN == IN_AOS) {
                const ulonglong2 row = reinterpret_cast<const ulonglong2 *>(src)[r];
                k[j] = row.x; v[j] = row.y;
            } else {
                k[j] = reinterpret_cast<const u64 *>(src)[r];
                v[j] = HAS_V ? reinterpret_cast<const u64 *>(src + HB_TILE * 8)[r] : 0ull;
            }
        }
        // The slot is refilled by the copy engine (async proxy) while these reads went through the generic
        // proxy: a proxy fence orders them before the release (without it ~1e-7 of the rows were read torn).
        fence_proxy_async();
        __syncwarp();
        if ((tid & 31u) == 0) mbar_arrive(&empty_bar[s]);   // this warp's rows are in registers: slot may be refilled
        if (!drain) ha_process_rows<OPK, TX, CACHE, HB_ROWS>(t, ctl, k, v, ok, tile * HB_TILE + tid, slot_out, hc_keys, hc_acc, use_cache, my_inserts, my_hits);
        if ((iter & 15u) == 15u) {   // periodic load-factor check (+ cache verdict); iter is CTA-uniform
            u32 w = __reduce_add_sync(0xffffffffu, my_inserts);
            my_inserts = 0;
            if ((tid & 31u) == 0 && w) atomicAdd(&s_inserts, w);
            if (CACHE && iter == 15u) {
                u32 hw = __reduce_add_sync(0xffffffffu, my_hits);
                if ((tid & 31u) == 0 && hw) atomicAdd(&s_hits, hw);
            }
            named_bar_sync(1, HA_THREADS);
            if (tid == 0) {
                u32 c = s_inserts;
                s_inserts = 0;
                u64 tot = atomicAdd(&ctl->n_inserted, (unsigned long long)c) + c;
                u32 ab = ld_volatile_u32(&ctl->abort);
                if (tot > max_inserts) { ab = 1; atomicExch(&ctl->abort, 1u); }
                s_abort = ab;
            }
            named_bar_sync(1, HA_THREADS);
            if (s_abort) drain = true;
            if (CACHE && iter == 15u && s_hits * 16u < 16u * HB_TILE) use_cache = false;
        }
    }
    // tail (< HB_TILE rows): plain loads, by the CTA whose turn it would have been
    if (!drain && (n % HB_TILE) && blockIdx.x == (u32)(n_full % gridDim.x)) {
        const u64 pol = policy_evict_first();
        const u64 base = n_full * HB_TILE;
        u64 k[HB_ROWS], v[HB_ROWS];
        bool ok[HB_ROWS];
#pragma unroll
        for (int j = 0; j < HB_ROWS; ++j) {
            const u64 idx = base + (u64)j * HA_THREADS + tid;
            ok[j] = idx < n;
            k[j] = 0; v[j] = 0;
            if (ok[j]) {
                if (IN == IN_AOS) { ulonglong2 r = ld_stream_u64x2(a + 2 * idx, pol); k[j] = r.x; v[j] = r.y; }
                else { k[j] = ld_stream_u64(a + idx, pol); if (HAS_V) v[j] = ld_stream_u64(b + idx, pol); }
            }
        }
        ha_process_rows<OPK, TX, CACHE, HB_ROWS>(t, ctl, k, v, ok, base + tid, slot_out, hc_keys, hc_acc, use_cache, my_inserts, my_hits);
    }
    if (CACHE) {   // flush the cache into the table (merge op)
        named_bar_sync(1, HA_THREADS);
        if (!drain)
            for (u32 i = tid; i < HC_SLOTS; i += HA_THREADS) {
                const u64 key = hc_keys[i];
                if (key == EMPTY_KEY) continue;
                const u64 hb = home_bucket(key, t.log_cap);
                u32 slot = 0;
                if (!table_resolve<OPK_FLUSH>(t, hb, ld_bucket(&t.keys[4 * hb]), key, hc_acc[i], slot, my_inserts)) atomicExch(&ctl->abort, 1u);
            }
    }
    u32 w = __reduce_add_sync(0xffffffffu, my_inserts);
    if ((tid & 31u) == 0 && w) atomicAdd(&s_inserts, w);
    named_bar_sync(1, HA_THREADS);
    if (tid == 0 && s_inserts) atomicAdd(&ctl->n_inserted, (unsigned long long)s_inserts);
}

// Strided key sample for the distinct-count estimate that sizes the first table.
template <int IN>
__global__ void sample_keys_kernel(const u64 *__restrict__ a, u64 n, u64 stride, u64 *__restrict__ out, u32 m)
{
    u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    u64 i = (u64)j * stride;
    if (i >= n) i = n - 1;
    out[j] = (IN == IN_AOS) ? a[2 * i] : a[i];
}

// Read-only lookup used by the join: slot index of `key`, or 0xFFFFFFFF.
VB_D u32 table_find(const Table &t, u64 key)
{
    const u64 cap = 1ull << t.log_cap, nb_mask = (cap >> 2) - 1;
    if (key == EMPTY_KEY) return t.keys[cap] == 1ull ? (u32)cap : 0xFFFFFFFFu;
    u64 b = home_bucket(key, t.log_cap);
    for (u32 probe = 0; probe <= HA_MAX_PROBE; ++probe) {
        const Bucket4 bk = ld_bucket(&t.keys[4 * b]);
        const int hit = bucket_find(bk, key);
        if (hit >= 0) return (u32)(4 * b + hit);
        if (bucket_find(bk, EMPTY_KEY) >= 0) return 0xFFFFFFFFu;
        b = (b + 1) & nb_mask;
    }
    return 0xFFFFFFFFu;
}

// ---------------------------------------------------------------------------------------------
// Radix pass (stable multisplit / one LSD digit)
// ---------------------------------------------------------------------------------------------
#ifndef VB_RP_TILE
#define VB_RP_TILE 4096
#endif
#ifndef VB_RPS_THREADS
#define VB_RPS_THREADS 512
#endif
constexpr int RP_THREADS = 256;
constexpr int RP_WARPS = RP_THREADS / 32;
constexpr int RP_TILE = VB_RP_TILE;              // rows per tile
constexpr int RP_ITEMS = RP_TILE / RP_THREADS;   // histogram kernel: items per thread per tile
constexpr int RP_NB = 256;                       // bins of an 8-bit pass (multisplit); bin NB = "invalid, drop"
constexpr int RPS_THREADS = VB_RPS_THREADS;      // scatter kernel: 16 warps x 8 items cover the same 4096-row tile with
constexpr int RPS_WARPS = RPS_THREADS / 32;      // <= 64 registers/thread, so 2 CTAs = 32 warps stay resident per SM
constexpr int RPS_ITEMS = RP_TILE / RPS_THREADS; // (256 x 16 needed 128 registers: 16 warps/SM, issue slots 32 % busy)
constexpr int RP_SORT_BITS = 8;                  // digit width of the LSD sort passes; a 10-bit variant was measured 2.4x slower per pass
                                                 // (per-tile scan over 1025 bins + 4-row write runs), profiles/r1_ops_10bit_digits.jsonl

enum : int { LD_SOA64 = 0, LD_AOS64 = 1, LD_KEY32_VAL_SOA = 2, LD_KEY32_VAL_AOS = 3, LD_TABLE_KV = 4, LD_TABLE_KI = 5 };

// Where a pass reads its rows from.  One struct, run-time mode (CTA-uniform branch).
struct Loader {
    int mode;
    const void *keys;   // u64* / u32* / rows (AoS) / table keys
    const void *vals;   // u64* (table modes: the accs array) or AoS rows for LD_KEY32_VAL_AOS
    u64 cap;            // table modes: number of regular slots (row `cap` is the special slot)
};

// Loader / digit modes are compile-time (LDM, DGM): a run-time switch per item left ptxas with a
// branch per load and no memory-level parallelism (profiles/r1_ncu_rp_before.txt).
template <typename KeyT, int LDM>
VB_D bool rp_load(const Loader &ld, u64 i, KeyT &key, u64 &val, u64 pol)
{
    if constexpr (LDM == LD_SOA64) {
        key = (KeyT)ld_stream_u64((const u64 *)ld.keys + i, pol);
        val = ld.vals ? ld_stream_u64((const u64 *)ld.vals + i, pol) : 0ull;
        return true;
    } else if constexpr (LDM == LD_AOS64) {
        ulonglong2 r = ld_stream_u64x2((const u64 *)ld.keys + 2 * i, pol);
        key = (KeyT)r.x; val = r.y;
        return true;
    } else if constexpr (LDM == LD_KEY32_VAL_SOA) {
        key = (KeyT)ld_stream_u32((const u32 *)ld.keys + i, pol);
        val = ld.vals ? ld_stream_u64((const u64 *)ld.vals + i, pol) : 0ull;
        return true;
    } else if constexpr (LDM == LD_KEY32_VAL_AOS) {
        key = (KeyT)ld_stream_u32((const u32 *)ld.keys + i, pol);
        val = ld_stream_u64((const u64 *)ld.vals + 2 * i + 1, pol);
        return true;
    } else {
        const u64 k = ld_stream_u64((const u64 *)ld.keys + i, pol);
        val = (LDM == LD_TABLE_KI) ? i : ld_stream_u64((const u64 *)ld.vals + i, pol);
        if (i == ld.cap) { key = (KeyT)EMPTY_KEY; return k == 1ull; }
        key = (KeyT)k;
        return k != EMPTY_KEY;
    }
}

// key only (histogram pass)
template <typename KeyT, int LDM>
VB_D bool rp_load_key(const Loader &ld, u64 i, KeyT &key, u64 pol)
{
    if constexpr (LDM == LD_SOA64) { key = (KeyT)ld_stream_u64((const u64 *)ld.keys + i, pol); return true; }
    else if constexpr (LDM == LD_AOS64) { key = (KeyT)ld_stream_u64((const u64 *)ld.keys + 2 * i, pol); return true; }
    else if constexpr (LDM == LD_KEY32_VAL_SOA || LDM == LD_KEY32_VAL_AOS) { key = (KeyT)ld_stream_u32((const u32 *)ld.keys + i, pol); return true; }
    else {
        const u64 k = ld_stream_u64((const u64 *)ld.keys + i, pol);
        if (i == ld.cap) { key = (KeyT)EMPTY_KEY; return k == 1ull; }
        key = (KeyT)k;
        return k != EMPTY_KEY;
    }
}

enum : int { DG_BITS = 0, DG_BUCKET = 1, DG_DEST = 2, DG_HASHTOP = 3 };

// Which bin a key goes to.  DG_BITS: radix digit of the (order-transformed) key.  DG_BUCKET:
// digit of HashPartitioner::get_partition(key).  DG_DEST: owning rank = partition % world.
// DG_HASHTOP: top bits of slot_hash(key) — pre-partitions rows so a table larger than L2 is visited region by region.
struct Digit {
    int mode;
    u32 shift, mask;
    int tx;
    u32 key_width;
    FastMod fm;        // % n_reduce
    FastMod fm_world;  // % world
};

template <typename KeyT, int DGM>
VB_D u32 rp_digit(const Digit &dg, KeyT key)
{
    if constexpr (DGM == DG_BITS) {
        u64 k = (sizeof(KeyT) == 8) ? tx_fwd((u64)key, dg.tx) : (u64)key;
        return (u32)(k >> dg.shift) & dg.mask;
    } else if constexpr (DGM == DG_HASHTOP) {
        // top bits of the table's slot hash: rows of one digit probe one contiguous region of the table
        return (u32)(slot_hash((u64)key) >> dg.shift) & dg.mask;
    } else {
        u32 b = get_partition((u64)key, dg.key_width, dg.fm);
        if constexpr (DGM == DG_DEST) return fastmod(b, dg.fm_world);
        return (b >> dg.shift) & dg.mask;
    }
}

// Lanes of the warp whose (BITS+1)-bit digit equals mine.  Built from BITS+1 ballots instead of
// MATCH.ANY: the hardware match iterates over the distinct values in the warp (~30 for random
// digits) and dominated both radix kernels (profiles/r1_ncu_rp_match_any.txt: short_scoreboard).
template <int BITS>
VB_D u32 warp_match_digit(u32 d)
{
    u32 peers = 0xffffffffu;
#pragma unroll
    for (int b = 0; b <= BITS; ++b) {          // BITS digit bits + the "invalid" bit
        const bool bit = (d >> b) & 1u;
        const u32 m = __ballot_sync(0xffffffffu, bit);
        peers &= bit ? m : ~m;
    }
    return peers;
}

// part p covers rows [p*rows_per_part, min(n, (p+1)*rows_per_part)); hist[d*num_parts + p].
// Each part is histogrammed by `split` CTAs (blockIdx.x = part*split + sub) that add their counts
// with global atomics, so the grid fills the machine even though there are only ~2 parts per SM.
// hist must be zeroed before the launch.
// Counting needs no ranking, so instead of a ballot match per item (78 instructions per item,
// math_pipe_throttle in profiles/r1_ncu_rp_ballot.txt) every LANE keeps private byte counters
// pc[warp][digit][lane] in shared memory: an item is one LDS.U8 / IADD / STS.U8, no atomics, no votes.
// A thread adds at most RP_ITEMS per tile, so the bytes are folded into the CTA's u32 histogram
// every 255 / RP_ITEMS tiles (15 * 16 = 240 <= 255).
constexpr size_t rp_hist_smem(int bits) { return (size_t)RP_WARPS * ((size_t)1 << bits) * 32; }

template <typename KeyT, int LDM, int DGM, int BITS>
__global__ void __launch_bounds__(RP_THREADS)
rp_hist_kernel(Loader ld, Digit dg, u64 n, u64 rows_per_part, u32 *__restrict__ hist, u32 num_parts, u32 split)
{
    constexpr int NB = 1 << BITS;
    extern __shared__ __align__(16) unsigned char pc_raw[];        // [RP_WARPS][NB][32] byte counters
    __shared__ u32 cta_hist[NB];
    const u32 tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    unsigned char *pc = pc_raw + (size_t)warp * NB * 32;
    u32 *pcw = (u32 *)pc;
    for (u32 i = lane; i < NB * 8; i += 32) pcw[i] = 0;
    for (u32 d = tid; d < NB; d += RP_THREADS) cta_hist[d] = 0;
    __syncthreads();
    const u64 pol = policy_evict_first();
    const u32 part = blockIdx.x / split, sub = blockIdx.x % split;
    const u64 begin = (u64)part * rows_per_part;
    const u64 end = min(n, begin + rows_per_part);
    auto fold = [&]() {      // warp-local: sum the 32 lane counters of each digit into cta_hist, clear them
        __syncwarp();
        for (u32 b = lane; b < NB; b += 32) {
            u32 s = 0;
#pragma unroll
            for (int w = 0; w < 8; ++w) {
                const u32 x = pcw[b * 8 + w];
                pcw[b * 8 + w] = 0;
                s += (x & 0xFF) + ((x >> 8) & 0xFF) + ((x >> 16) & 0xFF) + (x >> 24);
            }
            if (s) atomicAdd(&cta_hist[b], s);
        }
        __syncwarp();
    };
    constexpr int HB = 8;   // items per batch: keeps the u64 instantiation at <= 64 registers
    u32 tiles_since_fold = 0;
    constexpr bool STREAM = (LDM == LD_SOA64 || LDM == LD_AOS64 || LDM == LD_KEY32_VAL_SOA || LDM == LD_KEY32_VAL_AOS);   // every row valid
    for (u64 t0 = begin + (u64)sub * RP_TILE; t0 < end; t0 += (u64)split * RP_TILE) {
        if (STREAM && t0 + RP_TILE <= end) {      // whole tile in range: no bounds checks, no branch around the counter update
#pragma unroll 1
            for (int h = 0; h < RP_ITEMS; h += HB) {
                KeyT key[HB];
#pragma unroll
                for (int i = 0; i < HB; ++i) {
                    const u64 idx = t0 + (u64)warp * (32 * RP_ITEMS) + (u64)(h + i) * 32 + lane;
                    rp_load_key<KeyT, LDM>(ld, idx, key[i], pol);
                }
#pragma unroll
                for (int i = 0; i < HB; ++i) pc[rp_digit<KeyT, DGM>(dg, key[i]) * 32 + lane] += 1;
            }
            if (++tiles_since_fold == 255 / RP_ITEMS) { fold(); tiles_since_fold = 0; }
            continue;
        }
#pragma unroll 1
        for (int h = 0; h < RP_ITEMS; h += HB) {
            KeyT key[HB];
            bool ok[HB];
#pragma unroll
            for (int i = 0; i < HB; ++i) {
                const u64 idx = t0 + (u64)warp * (32 * RP_ITEMS) + (u64)(h + i) * 32 + lane;
                key[i] = 0;
                ok[i] = (idx < end) && rp_load_key<KeyT, LDM>(ld, idx, key[i], pol);
            }
#pragma unroll
            for (int i = 0; i < HB; ++i) {
                if (ok[i]) {
                    const u32 d = rp_digit<KeyT, DGM>(dg, key[i]);
                    pc[d * 32 + lane] += 1;      // private to this lane: plain read-modify-write
                }
            }
        }
        if (++tiles_since_fold == 255 / RP_ITEMS) { fold(); tiles_since_fold = 0; }
    }
    fold();
    __syncthreads();
    for (u32 d = tid; d < NB; d += RP_THREADS) {
        const u32 s = cta_hist[d];
        if (s) atomicAdd(&hist[(u64)d * num_parts + part], s);
    }
}

// Exclusive scan of hist[0 .. len) in place (single CTA); total written to hist[len].
__global__ void __launch_bounds__(1024) rp_scan_kernel(u32 *hist, u32 len)
{
    __shared__ u32 warp_sums[32];
    __shared__ u32 s_total;
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    const u32 per = (len + 1023u) / 1024u;
    const u32 lo = min(len, tid * per), hi = min(len, lo + per);
    u32 s = 0;
    for (u32 i = lo; i < hi; ++i) s += hist[i];
    u32 incl = s;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= (u32)off) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        u32 ws = warp_sums[lane];
        u32 wi = ws;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            u32 t = __shfl_up_sync(0xffffffffu, wi, off);
            if (lane >= (u32)off) wi += t;
        }
        warp_sums[lane] = wi - ws;
        if (lane == 31) s_total = wi;
    }
    __syncthreads();
    u32 run = warp_sums[warp] + (incl - s);
    for (u32 i = lo; i < hi; ++i) {
        u32 c = hist[i];
        hist[i] = run;
        run += c;
    }
    if (tid == 0) hist[len] = s_total;
}

// One stable scatter pass.  Per 4096-row tile: rank every row inside its warp by digit (ballots), scan
// the warp counts across the CTA, stage the tile in shared memory in output order together with each
// row's GLOBAL output index, then write it out with consecutive threads touching consecutive staged
// rows (runs of ~16 rows per digit → coalesced 64-128 B segments).  5 barriers per tile; the counters
// for the next tile are cleared and its loads are in flight while the current tile is written out.
// Destination tables of a REMOTE scatter: digit d (= destination rank) is written to the peer's
// receive arena mapped into this process (CUDA IPC over NVLink), at row adj[d] + flat_index.
struct RemoteDst {
    u64 *const *keys;   // [world] device array of peer key bases
    u64 *const *vals;   // [world]
    const u32 *adj;     // [world] (my row offset inside the peer's arena) - (start of digit d in the flat order)
    u32 world;
};

// REMOTE = the shuffle's exchange fused into the partition pass: instead of packing rows by
// destination rank locally and handing the buffers to an all-to-all, the staged runs are stored straight
// into the destination GPUs' HBM (st.global on peer-mapped addresses), so the NVLink transfer overlaps
// ranking/staging of the following tiles.
template <typename KeyT, bool HAS_VAL, int LDM, int DGM, int BITS, bool REMOTE = false>
__global__ void __launch_bounds__(RPS_THREADS, (RPS_THREADS > 512 ? 1 : RPS_THREADS > 256 ? 2 : 4))
rp_scatter_kernel(Loader ld, Digit dg, u64 n, u64 rows_per_part, const u32 *__restrict__ part_off, u32 num_parts,
                  KeyT *__restrict__ out_keys, u64 *__restrict__ out_vals, RemoteDst rd)
{
    constexpr int NB = 1 << BITS;
    static_assert(NB <= RPS_THREADS, "one thread per digit in the tile scan");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    u64 *stage_vals = (u64 *)smem_raw;                                       // [RP_TILE] if HAS_VAL
    KeyT *stage_keys = (KeyT *)(smem_raw + (HAS_VAL ? RP_TILE * 8 : 0));     // [RP_TILE]
    // the widest rows (u64 key + u64 value) stage the 1-byte digit and look the offset up at write-out
    // instead of staging a 4-byte output index: 18 % faster for them, 2-4 % slower for the others (A/B on B200)
    constexpr bool STAGE_IDX = !(sizeof(KeyT) == 8 && HAS_VAL);
    u32 *stage_out = (u32 *)(stage_keys + RP_TILE);                          // [RP_TILE] global output index (STAGE_IDX)
    unsigned char *stage_dig = (unsigned char *)(stage_keys + RP_TILE);      // [RP_TILE] digit (!STAGE_IDX)
    __shared__ u32 cnt[RPS_WARPS][NB + 1];   // per warp: count, then exclusive prefix over warps
    __shared__ u32 dbase[NB + 1];            // tile-local start of digit d; dbase[NB] = #valid rows of the tile
    __shared__ u32 gbase[NB + 1];            // run_off[d] - dbase[d]: staged position p of digit d goes to gbase[d] + p
    __shared__ u32 run_off[NB];              // global output offset of the next row of digit d for this part
    __shared__ u32 wtot[RPS_WARPS];
    __shared__ u64 *s_dk[REMOTE ? NB : 1];
    __shared__ u64 *s_dv[REMOTE ? NB : 1];
    __shared__ u32 s_adj[REMOTE ? NB : 1];
    static_assert(!REMOTE || (sizeof(KeyT) == 8 && HAS_VAL), "remote scatter moves (u64 key, u64 value) rows");
    if (REMOTE)
        for (u32 d = threadIdx.x; d < rd.world && d < (u32)NB; d += RPS_THREADS) { s_dk[d] = rd.keys[d]; s_dv[d] = rd.vals[d]; s_adj[d] = rd.adj[d]; }

    const u32 tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
    const u32 lt = lanemask_lt();
    const u64 pol = policy_evict_first();
    const u32 part = blockIdx.x;
    const u64 begin = (u64)part * rows_per_part;
    const u64 end = min(n, begin + rows_per_part);
    for (u32 d = tid; d < NB; d += RPS_THREADS) run_off[d] = part_off[(u64)d * num_parts + part];
    for (u32 d = tid; d < RPS_WARPS * (NB + 1); d += RPS_THREADS) (&cnt[0][0])[d] = 0;

    KeyT key[RPS_ITEMS];
    u64 val[RPS_ITEMS];
    bool ok[RPS_ITEMS];
    auto load_tile = [&](u64 t0) {
#pragma unroll
        for (int i = 0; i < RPS_ITEMS; ++i) {   // every load of the tile is issued before any is used
            const u64 idx = t0 + (u64)warp * (32 * RPS_ITEMS) + (u64)i * 32 + lane;
            key[i] = 0; val[i] = 0;
            ok[i] = (idx < end) && rp_load<KeyT, LDM>(ld, idx, key[i], val[i], pol);
        }
    };
    // (u64 key + u64 value needs 32 registers for the tile alone: prefetching spilled under the 64-register cap)
    constexpr bool PREFETCH = !(sizeof(KeyT) == 8 && HAS_VAL);
    if (PREFETCH && begin < end) load_tile(begin);
    __syncthreads();

    for (u64 t0 = begin; t0 < end; t0 += RP_TILE) {
        if (!PREFETCH) load_tile(t0);
        unsigned short dig[RPS_ITEMS], rank[RPS_ITEMS];
#pragma unroll
        for (int i = 0; i < RPS_ITEMS; ++i) dig[i] = (unsigned short)(ok[i] ? rp_digit<KeyT, DGM>(dg, key[i]) : (u32)NB);
#pragma unroll
        for (int i = 0; i < RPS_ITEMS; ++i) {
            const u32 d = dig[i];
            const u32 peers = warp_match_digit<BITS>(d);
            const u32 leader = (u32)(__ffs(peers) - 1);
            u32 base = 0;
            if (lane == leader) { base = cnt[warp][d]; cnt[warp][d] = base + __popc(peers); }   // only the group leader touches smem
            base = __shfl_sync(0xffffffffu, base, leader);
            rank[i] = (unsigned short)(base + __popc(peers & lt));
            __syncwarp();                                                       // orders this round's store before the next round's load
        }
        __syncthreads();                                                        // B1: warp counts complete
        // thread d < NB: exclusive scan of digit d over the warps, then a block-wide exclusive scan over the digits;
        // the "invalid" bin NB sits after all valid rows and is handled by one extra thread below
        u32 total = 0;
        if (tid < NB) {
#pragma unroll
            for (int w = 0; w < RPS_WARPS; ++w) { const u32 c = cnt[w][tid]; cnt[w][tid] = total; total += c; }
        }
        u32 incl = total;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= (u32)off) incl += t;
        }
        if (lane == 31) wtot[warp] = incl;
        __syncthreads();                                                        // B2: warp totals visible
        if (tid < NB) {
            u32 excl = incl - total;
            for (u32 w = 0; w < warp; ++w) excl += wtot[w];
            dbase[tid] = excl;
#pragma unroll
            for (int w = 0; w < RPS_WARPS; ++w) cnt[w][tid] += excl;            // cnt[w][d] = tile position of warp w's first row of digit d
            const u32 ro = run_off[tid];
            gbase[tid] = ro - excl;
            run_off[tid] = ro + total;
            if (tid == NB - 1) {                                                // rows of the invalid bin follow the valid ones
                u32 nv = excl + total;
                dbase[NB] = nv;
                for (int w = 0; w < RPS_WARPS; ++w) { const u32 c = cnt[w][NB]; cnt[w][NB] = nv; nv += c; }
            }
        }
        __syncthreads();                                                        // B3: positions / gbase visible
#pragma unroll
        for (int i = 0; i < RPS_ITEMS; ++i) {
            const u32 d = dig[i];
            const u32 pos = cnt[warp][d] + rank[i];
            stage_keys[pos] = key[i];
            if (HAS_VAL) stage_vals[pos] = val[i];
            if (d < NB) {                                   // rows with d == NB (invalid) sit past n_valid
                if (STAGE_IDX) stage_out[pos] = gbase[d] + pos;
                else stage_dig[pos] = (unsigned char)d;
            }
        }
        if (PREFETCH && t0 + RP_TILE < end) load_tile(t0 + RP_TILE);             // in flight during the write-out below
        __syncthreads();                                                        // B4: tile staged, cnt free
        for (u32 d = tid; d < RPS_WARPS * (NB + 1); d += RPS_THREADS) (&cnt[0][0])[d] = 0;
        const u32 n_valid = dbase[NB];
        for (u32 p = tid; p < n_valid; p += RPS_THREADS) {
            if (REMOTE) {
                const u32 d = stage_dig[p];
                const u32 o = gbase[d] + p + s_adj[d];
                s_dk[d][o] = (u64)stage_keys[p];
                s_dv[d][o] = stage_vals[p];
            } else {
                // (writing the same bytes to sequential destinations instead is only 0-5 % faster: the
                //  scattered DRAM writes are not what bounds this kernel — barriers and latency are)
                const u32 o = STAGE_IDX ? stage_out[p] : gbase[stage_dig[p]] + p;
                out_keys[o] = stage_keys[p];
                if (HAS_VAL) out_vals[o] = stage_vals[p];
            }
        }
        __syncthreads();                                                        // B5: staging buffers and cnt reusable
    }
}

template <typename KeyT, bool HAS_VAL, int BITS>
constexpr size_t rp_scatter_smem() { return (size_t)RP_TILE * ((HAS_VAL ? 8 : 0) + sizeof(KeyT) + ((sizeof(KeyT) == 8 && HAS_VAL) ? 1 : 4)); }

// ---------------------------------------------------------------------------------------------
// Unordered multisplit of the occupied slots of a combined table (reduce ops): (key, combiner) rows by reduce
// partition or by owner rank.  The reference's order inside a reduce partition is HashMap order (unspecified), so
// no stability is needed here: two small kernels (count, scatter with one global cursor claim per tile and bin)
// replace the histogram + single-CTA scan + stable scatter of the general pass, whose fixed cost (~150 us) is
// most of a step's seal/exchange time once the map-side combine has shrunk 1e9 rows to 1e6.
// ---------------------------------------------------------------------------------------------
constexpr int TS_THREADS = 256, TS_ITEMS = 8, TS_TILE = TS_THREADS * TS_ITEMS, TS_MAX_BINS = 256;

template <int DGM>
VB_D bool ts_load(const u64 *__restrict__ keys, u64 cap, u64 i, const Digit &dg, u64 &key, u32 &bin)
{
    if (i > cap) return false;
    const u64 k = keys[i];
    if (i == cap) { if (k != 1ull) return false; key = EMPTY_KEY; }      // special slot: a real key equal to the empty marker
    else { if (k == EMPTY_KEY) return false; key = k; }
    bin = rp_digit<u64, DGM>(dg, key);
    return true;
}

template <int DGM>
__global__ void __launch_bounds__(TS_THREADS) table_bin_count_kernel(const u64 *__restrict__ keys, u64 cap, Digit dg, u32 *__restrict__ counts)
{
    __shared__ u32 h[TS_MAX_BINS];
    for (u32 d = threadIdx.x; d < TS_MAX_BINS; d += TS_THREADS) h[d] = 0;
    __syncthreads();
    const u64 stride = (u64)gridDim.x * TS_THREADS;
    for (u64 i = (u64)blockIdx.x * TS_THREADS + threadIdx.x; i <= cap; i += stride) {
        u64 key; u32 bin;
        if (ts_load<DGM>(keys, cap, i, dg, key, bin)) atomicAdd(&h[bin], 1u);
    }
    __syncthreads();
    for (u32 d = threadIdx.x; d < TS_MAX_BINS; d += TS_THREADS) if (h[d]) atomicAdd(&counts[d], h[d]);
}

template <int DGM>
__global__ void __launch_bounds__(TS_THREADS)
table_bin_scatter_kernel(const u64 *__restrict__ keys, const u64 *__restrict__ accs, u64 cap, Digit dg, const u32 *__restrict__ counts,
                         u32 *__restrict__ cursors, u64 *__restrict__ out_keys, u64 *__restrict__ out_vals)
{
    __shared__ u32 base[TS_MAX_BINS], tile_cnt[TS_MAX_BINS], tile_base[TS_MAX_BINS], ws[TS_THREADS / 32];
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    {   // exclusive scan of the global counts (every CTA redoes these 256 adds instead of a separate scan kernel)
        const u32 c = counts[tid];
        u32 incl = c;
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= (u32)off) incl += t; }
        if (lane == 31) ws[warp] = incl;
        __syncthreads();
        u32 b = 0;
        for (u32 w = 0; w < warp; ++w) b += ws[w];
        base[tid] = b + incl - c;
        tile_cnt[tid] = 0;
    }
    __syncthreads();
    const u64 n_tiles = (cap + 1 + TS_TILE - 1) / TS_TILE;
    for (u64 tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        u64 key[TS_ITEMS], val[TS_ITEMS];
        u32 br[TS_ITEMS];                         // bin | local rank << 8 ; 0xFFFFFFFF = no row
#pragma unroll
        for (int j = 0; j < TS_ITEMS; ++j) {
            const u64 i = tile * TS_TILE + (u64)j * TS_THREADS + tid;
            u32 bin;
            br[j] = 0xFFFFFFFFu;
            if (ts_load<DGM>(keys, cap, i, dg, key[j], bin)) {
                val[j] = accs[i];
                br[j] = bin | (atomicAdd(&tile_cnt[bin], 1u) << 8);
            }
        }
        __syncthreads();
        { const u32 c = tile_cnt[tid]; if (c) tile_base[tid] = base[tid] + atomicAdd(&cursors[tid], c); }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < TS_ITEMS; ++j) {
            if (br[j] == 0xFFFFFFFFu) continue;
            const u32 o = tile_base[br[j] & 0xFFu] + (br[j] >> 8);
            out_keys[o] = key[j];
            out_vals[o] = val[j];
        }
        tile_cnt[tid] = 0;
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Generic multi-block exclusive scan (u64), chunk = 4096 elements per CTA
// ---------------------------------------------------------------------------------------------
constexpr int SC_THREADS = 256;
constexpr int SC_ITEMS = 16;
constexpr int SC_CHUNK = SC_THREADS * SC_ITEMS;

VB_D u64 block_exclusive_scan_u64(u64 v, u64 *total, u64 *warp_sums /*[8]*/)
{
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    u64 incl = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        u64 t = __shfl_up_sync(0xffffffffu, incl, off);
        if (lane >= (u32)off) incl += t;
    }
    if (lane == 31) warp_sums[warp] = incl;
    __syncthreads();
    u64 wbase = 0, tsum = 0;
#pragma unroll
    for (int w = 0; w < SC_THREADS / 32; ++w) {
        u64 x = warp_sums[w];
        if ((u32)w < warp) wbase += x;
        tsum += x;
    }
    *total = tsum;
    __syncthreads();
    return wbase + incl - v;
}

__global__ void __launch_bounds__(SC_THREADS) scan_reduce_kernel(const u64 *__restrict__ in, u64 n, u64 *__restrict__ sums)
{
    __shared__ u64 ws[SC_THREADS / 32];
    const u64 base = (u64)blockIdx.x * SC_CHUNK;
    u64 s = 0;
    for (int i = 0; i < SC_ITEMS; ++i) {
        u64 idx = base + (u64)i * SC_THREADS + threadIdx.x;
        if (idx < n) s += in[idx];
    }
    u64 tot;
    block_exclusive_scan_u64(s, &tot, ws);
    if (threadIdx.x == 0) sums[blockIdx.x] = tot;
}

// out[i] = offsets[block] + exclusive prefix within the chunk.  offsets may be NULL (single chunk).
// If total_out != NULL the last block writes the grand total there.
__global__ void __launch_bounds__(SC_THREADS)
scan_apply_kernel(const u64 *__restrict__ in, u64 *__restrict__ out, u64 n, const u64 *__restrict__ offsets, u64 *total_out)
{
    __shared__ u64 ws[SC_THREADS / 32];
    const u64 base = (u64)blockIdx.x * SC_CHUNK + (u64)threadIdx.x * SC_ITEMS;
    u64 v[SC_ITEMS];
    u64 s = 0;
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i) {
        v[i] = (base + i < n) ? in[base + i] : 0ull;
        s += v[i];
    }
    u64 tot;
    u64 run = block_exclusive_scan_u64(s, &tot, ws) + (offsets ? offsets[blockIdx.x] : 0ull);
    const u64 carry_in = offsets ? offsets[blockIdx.x] : 0ull;
#pragma unroll
    for (int i = 0; i < SC_ITEMS; ++i) {
        if (base + i < n) out[base + i] = run;
        run += v[i];
    }
    if (total_out && blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) *total_out = carry_in + tot;
}

// ---------------------------------------------------------------------------------------------
// group_by_key helpers
// ---------------------------------------------------------------------------------------------
// dense_of_slot[cslot[j]] = j   (cslot holds slot indices as u64 payloads of the bucket multisplit)
__global__ void scatter_dense_kernel(const u64 *__restrict__ cslot, u32 n, u32 *__restrict__ dense_of_slot)
{
    u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) dense_of_slot[cslot[j]] = j;
}

// ids[i] = dense_of_slot[ids[i]] in place (the 4 MB–64 MB dense_of_slot array is L2-resident)
__global__ void translate_ids_kernel(u32 *__restrict__ ids, u64 n, const u32 *__restrict__ dense_of_slot)
{
    // One look-up per thread and iteration, 2048 threads per SM: 4.4 ms for 1e9 ids, against a floor of 3.5 ms (one L2 request per
    // id at the 2.87e11/s the chip sustains).  Tried and slower (profiles/r2_group_glue_tried.txt): fusing the look-up into the first
    // sort pass's histogram kernel (8.5 ms instead of 4.4 + 1.3: 24 warps per SM cannot cover two dependent L2 round trips per
    // batch), and four ids per thread with evict-first look-ups (6.1 ms: the hint ages the table out of L2).
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (; i < n; i += stride) ids[i] = dense_of_slot[ids[i]];
}

// CSR offsets from sorted dense ids: offsets[id] = first row of id; offsets[n_ids] = n.
__global__ void csr_bounds_kernel(const u32 *__restrict__ ids, u64 n, u64 *__restrict__ offsets, u64 n_ids)
{
    // four ids per thread (one 128-bit load + the id just before them): 2.5x fewer load instructions than one id per thread
    const u64 n4 = n / 4;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    const u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (t == 0) offsets[n_ids] = n;
    for (u64 j = t; j < n4; j += stride) {
        const uint4 v = reinterpret_cast<const uint4 *>(ids)[j];
        const u64 i = 4 * j;
        const u32 prev = j ? ids[i - 1] : ~v.x;          // j == 0: anything different from v.x
        if (prev != v.x) offsets[v.x] = i;
        if (v.x != v.y) offsets[v.y] = i + 1;
        if (v.y != v.z) offsets[v.z] = i + 2;
        if (v.z != v.w) offsets[v.w] = i + 3;
    }
    for (u64 i = 4 * n4 + t; i < n; i += stride) {       // the last n % 4 ids
        const u32 id = ids[i];
        if (i == 0 || ids[i - 1] != id) offsets[id] = i;
    }
}

// out[i] = tx_inv(in[i])
__global__ void tx_inv_kernel(u64 *__restrict__ v, u64 n, int tx)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = tx_inv(v[i], tx);
}

// de-interleave AoS rows into SoA (gather of map partitions that are not contiguous)
__global__ void aos_to_soa_kernel(const u64 *__restrict__ rows, u64 n, u64 *__restrict__ keys, u64 *__restrict__ vals)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    const u64 pol = policy_evict_first();
    for (; i < n; i += stride) {
        ulonglong2 r = ld_stream_u64x2(rows + 2 * i, pol);
        keys[i] = r.x;
        vals[i] = r.y;
    }
}

// ---------------------------------------------------------------------------------------------
// join (CoGroupedRdd::compute + cross product)
// ---------------------------------------------------------------------------------------------
// For left keys [lb, le): find the key in the right shuffle's dictionary; cnt = lenL * lenR.
__global__ void join_probe_kernel(const u64 *__restrict__ lkeys, const u64 *__restrict__ loffs, u32 lb, u32 le,
                                  Table rtab, const u32 *__restrict__ r_dense,
                                  const u64 *__restrict__ roffs, u64 *__restrict__ cnt, u32 *__restrict__ match)
{
    u32 j = lb + blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= le) return;
    u64 key = lkeys[j];
    u32 s = table_find(rtab, key);
    u64 c = 0;
    u32 m = 0xFFFFFFFFu;
    if (s != 0xFFFFFFFFu) {
        m = r_dense[s];
        c = (loffs[j + 1] - loffs[j]) * (roffs[m + 1] - roffs[m]);
    }
    cnt[j - lb] = c;
    match[j - lb] = m;
}

// One thread per output row: binary-search the owning left key, then (v, w) = divmod.
__global__ void join_expand_kernel(const u64 *__restrict__ pos /*[nl] exclusive*/, u32 nl, u64 total,
                                   const u64 *__restrict__ lkeys, const u64 *__restrict__ loffs, const u64 *__restrict__ lvals,
                                   u32 lb, const u32 *__restrict__ match, const u64 *__restrict__ roffs,
                                   const u64 *__restrict__ rvals, u64 *__restrict__ out_k, u64 *__restrict__ out_v,
                                   u64 *__restrict__ out_w)
{
    u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (; o < total; o += stride) {
        u32 lo = 0, hi = nl;   // largest j with pos[j] <= o  (keys with cnt 0 share pos with the next)
        while (hi - lo > 1) {
            u32 mid = (lo + hi) >> 1;
            if (pos[mid] <= o) lo = mid; else hi = mid;
        }
        const u32 j = lo;
        const u32 m = match[j];
        const u64 local = o - pos[j];
        const u64 lenr = roffs[m + 1] - roffs[m];
        const u64 vi = local / lenr, wi = local - vi * lenr;
        out_k[o] = lkeys[lb + j];
        out_v[o] = lvals[loffs[lb + j] + vi];
        out_w[o] = rvals[roffs[m] + wi];
    }
}

// ---------------------------------------------------------------------------------------------
// cogroup / outer joins (CoGroupedRdd::compute, co_grouped_rdd.rs:206-249): the union of the key sets of one
// partition, in union order — first the nl left keys in left CSR order (union key u is left key lb + u, match[u]
// its right dense id or CG_NONE), then the right keys no left key matched, in right CSR order (ronly[u - nl]).
// ---------------------------------------------------------------------------------------------
constexpr u32 CG_NONE = 0xFFFFFFFFu;
enum : int { CG_LEFT = 1, CG_RIGHT = 2 };   // the sides an outer join keeps when the other one is empty (VB_JOIN_* bits)

// join_probe_kernel for one partition, plus: the right key it hits is no longer right-only (ronly_flag[m - rb] = 0)
__global__ void cogroup_probe_kernel(const u64 *__restrict__ lkeys, u32 lb, u32 nl, Table rtab, const u32 *__restrict__ r_dense,
                                     u32 rb, u32 re, u32 *__restrict__ match, unsigned char *__restrict__ ronly_flag)
{
    const u32 j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= nl) return;
    const u32 s = table_find(rtab, lkeys[lb + j]);
    u32 m = CG_NONE;
    if (s != 0xFFFFFFFFu) {
        m = r_dense[s];
        if (m >= rb && m < re) ronly_flag[m - rb] = 0;
        else m = CG_NONE;
    }
    match[j] = m;
}

// value counts of union key u on both sides and its right dense id (CG_NONE: no right values)
VB_D void cogroup_key(u32 u, u32 nl, u32 lb, const u64 *__restrict__ loffs, const u32 *__restrict__ match,
                      const u32 *__restrict__ ronly, const u64 *__restrict__ roffs, u64 &lc, u64 &rc, u32 &m)
{
    if (u < nl) { lc = loffs[lb + u + 1] - loffs[lb + u]; m = match[u]; }
    else { lc = 0; m = ronly[u - nl]; }
    rc = m != CG_NONE ? roffs[m + 1] - roffs[m] : 0;
}

// largest u < nu with pos[u] <= o (union keys without output share pos with the next one)
VB_D u32 cogroup_owner(const u64 *__restrict__ pos, u32 nu, u64 o)
{
    u32 lo = 0, hi = nu;
    while (hi - lo > 1) {
        const u32 mid = (lo + hi) >> 1;
        if (pos[mid] <= o) lo = mid; else hi = mid;
    }
    return lo;
}

// per union key: left / right value counts (cnt_l / cnt_r, may be NULL) and output rows under an outer `kind` (cnt_rows, may be NULL)
__global__ void cogroup_count_kernel(u32 nl, u32 nu, u32 lb, const u64 *__restrict__ loffs, const u32 *__restrict__ match,
                                     const u32 *__restrict__ ronly, const u64 *__restrict__ roffs, int kind,
                                     u64 *__restrict__ cnt_l, u64 *__restrict__ cnt_r, u64 *__restrict__ cnt_rows)
{
    const u32 u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nu) return;
    u64 lc, rc;
    u32 m;
    cogroup_key(u, nl, lb, loffs, match, ronly, roffs, lc, rc, m);
    if (cnt_l) cnt_l[u] = lc;
    if (cnt_r) cnt_r[u] = rc;
    if (cnt_rows) cnt_rows[u] = (lc && rc) ? lc * rc : lc ? ((kind & CG_LEFT) ? lc : 0) : ((kind & CG_RIGHT) ? rc : 0);
}

// out[nl + i] = rkeys[ronly[i]]: the right-only keys after the left key slice
__global__ void cogroup_keys_kernel(const u32 *__restrict__ ronly, u32 nro, const u64 *__restrict__ rkeys, u64 *__restrict__ out)
{
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nro) out[i] = rkeys[ronly[i]];
}

// One thread per right value in union order: binary-search the owning union key in the scanned right counts.
__global__ void cogroup_gather_right_kernel(const u64 *__restrict__ offs_r /*[nu+1], partition-local*/, u32 nu, u64 total, u32 nl,
                                            const u32 *__restrict__ match, const u32 *__restrict__ ronly,
                                            const u64 *__restrict__ roffs, const u64 *__restrict__ rvals, u64 *__restrict__ out)
{
    u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (; o < total; o += stride) {
        const u32 u = cogroup_owner(offs_r, nu, o);
        const u32 m = u < nl ? match[u] : ronly[u - nl];
        out[o] = rvals[roffs[m] + (o - offs_r[u])];
    }
}

// One thread per outer-join row: binary-search the owning union key, then (v, w) in v-major order; an absent side is
// written as 0 with its bit clear in valid (1 = v present, 2 = w present).
__global__ void outer_expand_kernel(const u64 *__restrict__ pos /*[nu] exclusive*/, u32 nu, u64 total, u32 nl, u32 lb,
                                    const u64 *__restrict__ lkeys, const u64 *__restrict__ loffs, const u64 *__restrict__ lvals,
                                    const u32 *__restrict__ match, const u32 *__restrict__ ronly, const u64 *__restrict__ rkeys,
                                    const u64 *__restrict__ roffs, const u64 *__restrict__ rvals, u64 *__restrict__ out_k,
                                    u64 *__restrict__ out_v, u64 *__restrict__ out_w, unsigned char *__restrict__ out_valid)
{
    u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (; o < total; o += stride) {
        const u32 u = cogroup_owner(pos, nu, o);
        u64 lc, rc;
        u32 m;
        cogroup_key(u, nl, lb, loffs, match, ronly, roffs, lc, rc, m);
        const u64 local = o - pos[u];
        u64 v = 0, w = 0;
        unsigned char valid;
        if (lc && rc) {
            const u64 vi = local / rc, wi = local - vi * rc;
            v = lvals[loffs[lb + u] + vi];
            w = rvals[roffs[m] + wi];
            valid = CG_LEFT | CG_RIGHT;
        } else if (lc) {
            v = lvals[loffs[lb + u] + local];
            valid = CG_LEFT;
        } else {
            w = rvals[roffs[m] + local];
            valid = CG_RIGHT;
        }
        out_k[o] = u < nl ? lkeys[lb + u] : rkeys[m];
        out_v[o] = v;
        out_w[o] = w;
        if (out_valid) out_valid[o] = valid;
    }
}

// ---------------------------------------------------------------------------------------------
// bincode 1.2.1 blob codec (SURVEY §8(f) N1): pure byte shuffling, HBM-bound
// ---------------------------------------------------------------------------------------------
// Vec<(u64,u64)>: out = u64 n | n x (k, c)
__global__ void blob_pairs_kernel(const u64 *__restrict__ keys, const u64 *__restrict__ comb, u64 n, u64 *__restrict__ out)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    if (i == 0) out[0] = n;
    for (; i < n; i += stride) {
        out[1 + 2 * i] = keys[i];
        out[2 + 2 * i] = comb ? comb[i] : 0ull;
    }
}

// Vec<(u64,Vec<u64>)>: record i starts at word 1 + 2 i + offs[i] - base: (k, len, values...)
__global__ void blob_group_kernel(const u64 *__restrict__ keys, const u64 *__restrict__ offs /*[nk+1], absolute*/, u64 nk,
                                  const u64 *__restrict__ vals /*absolute index*/, u64 *__restrict__ out)
{
    const u64 base = offs[0], nv = offs[nk] - base;
    u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    if (t == 0) out[0] = nk;
    for (u64 i = t; i < nk; i += stride) {
        const u64 w = 1 + 2 * i + (offs[i] - base);
        out[w] = keys[i];
        out[w + 1] = offs[i + 1] - offs[i];
    }
    for (u64 j = t; j < nv; j += stride) {      // value j belongs to the key i with offs[i] <= base + j < offs[i+1]
        u64 lo = 0, hi = nk;
        while (hi - lo > 1) {
            const u64 mid = (lo + hi) >> 1;
            if (offs[mid] - base <= j) lo = mid; else hi = mid;
        }
        out[1 + 2 * (lo + 1) + j] = vals[base + j];
    }
}

// OR and AND over all (order-transformed) keys: a radix digit on which every key agrees needs no pass.
__global__ void key_bits_kernel(const u64 *__restrict__ keys, u64 stride_words, u64 n, int tx, unsigned long long *__restrict__ out /*[2]: or, and*/)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 step = (u64)gridDim.x * blockDim.x;
    const u64 pol = policy_evict_first();
    u64 o = 0, a = ~0ull;
    for (; i < n; i += step) {
        const u64 k = tx_fwd(ld_stream_u64(keys + i * stride_words, pol), tx);
        o |= k; a &= k;
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) {
        o |= __shfl_xor_sync(0xffffffffu, o, off);
        a &= __shfl_xor_sync(0xffffffffu, a, off);
    }
    if ((threadIdx.x & 31u) == 0) { atomicOr(&out[0], (unsigned long long)o); atomicAnd(&out[1], (unsigned long long)a); }
}

// ---------------------------------------------------------------------------------------------
// sort_by_key partition cuts: start of partition p = floor(p*n/R) moved past equal keys
// ---------------------------------------------------------------------------------------------
__global__ void sort_cuts_kernel(const u64 *__restrict__ keys, u64 n, u32 n_parts, u64 *__restrict__ starts)
{
    u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p > n_parts) return;
    if (p == 0) { starts[0] = 0; return; }
    if (p == n_parts) { starts[p] = n; return; }
    u64 c = ((u64)p * n) / n_parts;   // n < 2^32 and p < 2^32: no overflow
    if (c > 0 && c < n && keys[c] == keys[c - 1]) {   // upper bound of keys[c-1] in [c, n)
        const u64 k = keys[c - 1];
        u64 lo = c, hi = n;
        while (lo < hi) {
            u64 mid = lo + ((hi - lo) >> 1);
            if (keys[mid] == k) lo = mid + 1; else hi = mid;
        }
        c = lo;
    }
    starts[p] = c;
}

// ---------------------------------------------------------------------------------------------
// Synthetic input (SURVEY.md §8(d)); must match oracle/vega_oracle.c:vo_gen_uniform bit for bit
// ---------------------------------------------------------------------------------------------
enum : int { GEN_UNIFORM = 0, GEN_ZIPF = 1, GEN_UNIQUE = 2 };

__global__ void gen_pairs_kernel(u64 *__restrict__ rows, u64 *__restrict__ keys, u64 *__restrict__ vals, u64 first, u64 n,
                                 int mode, u64 n_distinct, u64 rank_base, u64 seed_k, u64 seed_v,
                                 const double *__restrict__ zipf_cdf)
{
    u64 t = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    for (; t < n; t += stride) {
        const u64 i = first + t;
        u64 rank;
        if (mode == GEN_UNIQUE) {
            rank = rank_base + i;
        } else if (mode == GEN_ZIPF) {
            const double u = (double)(splitmix64(seed_k + i) >> 11) * (1.0 / 9007199254740992.0);
            u64 lo = 0, hi = n_distinct - 1;     // first index with cdf[idx] >= u
            while (lo < hi) {
                u64 mid = (lo + hi) >> 1;
                if (zipf_cdf[mid] >= u) hi = mid; else lo = mid + 1;
            }
            rank = lo;
        } else {
            rank = splitmix64(seed_k + i) % n_distinct;
        }
        const u64 k = splitmix64(rank ^ 0xA5A5A5A5A5A5A5A5ull);
        const u64 v = splitmix64(seed_v + i) & 0xFFFFFull;
        if (rows) {
            ulonglong2 r; r.x = k; r.y = v;
            *reinterpret_cast<ulonglong2 *>(rows + 2 * t) = r;
        } else {
            keys[t] = k;
            if (vals) vals[t] = v;
        }
    }
}

}  // namespace vb
