// engine.cu — C ABI of libvega_b200.so (see include/vega_b200.h) and the host orchestration of
// the shuffle + aggregation kernels in kernels.cuh.  sm_100a only; no CPU fallback: every
// compute entry needs a CUDA device and fails with VB_ERR_CUDA otherwise.
#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/vega_b200.h"
#include "kernels.cuh"
#include "sweep.cuh"
#include "gsweep.cuh"
#include <type_traits>

using namespace vb;

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int set_err(int code, const char *fmt, ...)
{
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

#define CU(expr)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (expr);                                                                        \
        if (e_ != cudaSuccess) {                                                                        \
            cudaGetLastError();                                                                         \
            return set_err(e_ == cudaErrorMemoryAllocation ? VB_ERR_OOM : VB_ERR_CUDA, "%s:%d %s: %s", \
                           __FILE__, __LINE__, #expr, cudaGetErrorString(e_));                          \
        }                                                                                               \
    } while (0)

#define TRY(expr)                  \
    do {                           \
        int rc_ = (expr);          \
        if (rc_ != VB_OK) return rc_; \
    } while (0)

extern "C" const char *vb_last_error(void) { return g_err.c_str(); }
extern "C" const char *vb_version(void) { return "vega_b200 0.1 sm_100a"; }

// ---------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------
enum { K_HASH_AGG = 0, K_DICT = 1, K_MERGE = 2, K_RP_HIST = 3, K_RP_SCAN = 4, K_RP_SCATTER = 5, K_MISC = 6, K_JOIN = 7, K_N = 8 };

struct vb_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;          // H2D staging copies (overlap the kernels on `stream`)
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_kernel[2] = {nullptr, nullptr}, ev_ready = nullptr;
    std::vector<void *> pinned_slots;            // 64-byte pinned cells for per-call D2H status words (free list)
    cudaMemPool_t pool = nullptr;
    std::mutex mu;                 // serialises device work of this context
    bool profile = false;
    void *h_scratch = nullptr;     // pinned, 1 MiB
    size_t h_scratch_bytes = 1 << 20;
    double *zipf_cdf = nullptr;    // cached device CDF for vb_gen_pairs
    u64 zipf_n = 0;
    double zipf_s = 0;
    std::map<const void *, int> occ_cache;
    // P2P exchange: this rank's receive arena (cudaMalloc'ed, exported with CUDA IPC) and the peers' arenas
    void *arena = nullptr;
    size_t arena_bytes = 0;
    u64 arena_gen = 0;
    struct Peer { void *base = nullptr; u64 gen = 0; bool self = false; };
    std::map<u32, Peer> peers;
    std::vector<void *> retired_arenas;   // outgrown arenas some peer may still have mapped: freed by vb_ctx_arena_release_retired
    struct Comm *comm = nullptr;          // NCCL communicator + exchange scratch (vb_ctx_comm_init)
};
static void comm_teardown(vb_ctx *c);

struct DevBuf {   // stream-ordered device allocation, freed on scope exit unless released
    vb_ctx *c = nullptr;
    void *p = nullptr;
    DevBuf() {}
    explicit DevBuf(vb_ctx *c_) : c(c_) {}
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { reset(); }
    void reset()
    {
        if (p) cudaFreeAsync(p, c->stream);
        p = nullptr;
    }
    int alloc(size_t bytes)
    {
        reset();
        if (bytes == 0) bytes = 16;
        CU(cudaMallocAsync(&p, bytes, c->pool, c->stream));
        return VB_OK;
    }
    template <typename T> T *as() const { return (T *)p; }
    void *release()
    {
        void *q = p;
        p = nullptr;
        return q;
    }
};

static void dev_free(vb_ctx *c, const void *p)
{
    if (p) cudaFreeAsync((void *)p, c->stream);
}

template <typename K>
static int occupancy(vb_ctx *c, K kernel, int threads, size_t smem)
{
    auto it = c->occ_cache.find((const void *)kernel);
    if (it != c->occ_cache.end()) return it->second;
    int nb = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, threads, smem) != cudaSuccess || nb < 1) {
        cudaGetLastError();
        nb = 1;
    }
    c->occ_cache[(const void *)kernel] = nb;
    return nb;
}

extern "C" int32_t vb_ctx_create(int32_t device_id, vb_ctx **out)
{
    if (!out) return set_err(VB_ERR_INVALID, "vb_ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_err(VB_ERR_CUDA, "vb_ctx_create: no CUDA device (%s); libvega_b200 has no CPU fallback",
                       e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    if (device_id < 0 || device_id >= ndev) return set_err(VB_ERR_INVALID, "vb_ctx_create: device %d of %d", device_id, ndev);
    CU(cudaSetDevice(device_id));
    vb_ctx *c = new vb_ctx();
    c->device = device_id;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device_id));
    c->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    // a private stream-ordered pool: the process-wide default pool (shared with any other cudaMallocAsync
    // user) is left untouched; ours keeps its memory between shuffles (steady-state steps never call
    // cudaMalloc) until vb_ctx_trim / vb_ctx_destroy
    cudaMemPoolProps pp;
    memset(&pp, 0, sizeof(pp));
    pp.allocType = cudaMemAllocationTypePinned;
    pp.handleTypes = cudaMemHandleTypeNone;
    pp.location.type = cudaMemLocationTypeDevice;
    pp.location.id = device_id;
    CU(cudaMemPoolCreate(&c->pool, &pp));
    uint64_t thr = ~0ull;
    CU(cudaMemPoolSetAttribute(c->pool, cudaMemPoolAttrReleaseThreshold, &thr));
    CU(cudaMallocHost(&c->h_scratch, c->h_scratch_bytes));
    CU(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        CU(cudaEventCreateWithFlags(&c->ev_copied[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c->ev_kernel[i], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&c->ev_ready, cudaEventDisableTiming));
    {   // the last 4 KiB of the pinned scratch page hold 64 status cells
        char *base = (char *)c->h_scratch + c->h_scratch_bytes - 4096;
        for (int i = 0; i < 64; ++i) c->pinned_slots.push_back(base + 64 * i);
    }
    *out = c;
    return VB_OK;
}

extern "C" int32_t vb_ctx_destroy(vb_ctx *c)
{
    if (!c) return VB_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    if (c->zipf_cdf) cudaFreeAsync(c->zipf_cdf, c->stream);
    cudaStreamSynchronize(c->stream);
    for (auto &kv : c->peers) if (kv.second.base && !kv.second.self) cudaIpcCloseMemHandle(kv.second.base);
    // An exported arena must outlive every importer's mapping (cudaFree of a region a peer still has open is
    // undefined): with a communicator, all ranks close their mappings above, meet at a barrier, then free.
    comm_teardown(c);
    for (void *p : c->retired_arenas) cudaFree(p);
    if (c->arena) cudaFree(c->arena);
    cudaFreeHost(c->h_scratch);
    cudaStreamSynchronize(c->copy_stream);
    cudaStreamDestroy(c->copy_stream);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(c->ev_copied[i]); cudaEventDestroy(c->ev_kernel[i]); }
    cudaEventDestroy(c->ev_ready);
    cudaStreamDestroy(c->stream);
    if (c->pool) cudaMemPoolDestroy(c->pool);
    delete c;
    return VB_OK;
}

extern "C" int32_t vb_ctx_trim(vb_ctx *c, uint64_t keep_bytes)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    CU(cudaMemPoolTrimTo(c->pool, (size_t)keep_bytes));
    return VB_OK;
}

extern "C" int32_t vb_ctx_synchronize(vb_ctx *c)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}

extern "C" int32_t vb_ctx_set_profile(vb_ctx *c, int32_t on)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    c->profile = on != 0;
    return VB_OK;
}

extern "C" int32_t vb_ctx_device(vb_ctx *c) { return c ? c->device : -1; }
extern "C" void *vb_ctx_stream(vb_ctx *c) { return c ? (void *)c->stream : nullptr; }

extern "C" int32_t vb_ctx_mem_info(vb_ctx *c, uint64_t *reserved, uint64_t *high_water)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    uint64_t r = 0, h = 0;
    CU(cudaMemPoolGetAttribute(c->pool, cudaMemPoolAttrReservedMemCurrent, &r));
    CU(cudaMemPoolGetAttribute(c->pool, cudaMemPoolAttrUsedMemHigh, &h));
    if (reserved) *reserved = r;
    if (high_water) *high_water = h;
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// shuffle state
// ---------------------------------------------------------------------------------------------
struct MapOut {
    bool present = false;
    u64 n_rows = 0;
    // reduce ops: the combined table of this map task (== SHUFFLE_CACHE[(sid, map, *)])
    void *table = nullptr;      // table_at(table, log_cap)
    u32 log_cap = 0;
    u64 n_inserted = 0;
    // group/sort ops: the rows (device), AoS or SoA
    const u64 *rows = nullptr;
    const u64 *keys = nullptr;
    const u64 *vals = nullptr;
    bool owned = false;
    bool in_shared = false;   // reduce ops, borrowed device input: combined straight into the shuffle's shared table
};

struct Timer {
    cudaEvent_t a, b;
    int klass;   // K_* or -1 (map call) / -2 (seal call)
    u64 rows;
};

struct JoinPlan {
    u64 total = 0;
    u32 nl = 0;
    u64 *pos = nullptr;
    u32 *match = nullptr;
};

// cogroup / outer joins of one partition: the union of both key sets (see cogroup_probe_kernel)
struct CogroupPlan {
    u32 nl = 0, nro = 0;       // left keys of the partition, right-only keys
    u32 *match = nullptr;      // [nl] right dense id of each left key, or CG_NONE
    u32 *ronly = nullptr;      // [nro] dense ids of the right-only keys, in right CSR order
    int kind = 0;              // outer-join kind whose row positions are cached (0 = none yet)
    u64 rows = 0;
    u64 *rowpos = nullptr;     // [nl + nro] exclusive scan of the output rows per union key under `kind`
};

struct vb_shuf {
    vb_ctx *ctx = nullptr;
    u64 id = 0;
    u32 n_map = 0, n_reduce = 0;
    int kdt = 0, vdt = 0, agg = 0, part = 0;
    u32 key_width = 8;
    u64 hint = 0;
    u64 learned_distinct = 0;      // distinct keys seen by the previous table build of this shuffle
    // Shared table of the map tasks whose input is VB_DEVICE_BORROWED (valid until seal): the named ops are
    // associative and commutative, so those tasks combine into ONE table, launched back to back without a
    // host round trip per task and without a merge at seal.  If it overflows, or a map id is resubmitted,
    // seal rebuilds it from the still-borrowed inputs (same restart logic as build_table).
    void *sh_tab = nullptr;
    u32 sh_log_cap = 0;
    TableCtl *sh_ctl = nullptr;
    u64 sh_max_inserts = 0;
    bool sh_dirty = false;
    u32 rank = 0, world = 1;
    std::vector<MapOut> maps;
    std::mutex mu;
    std::condition_variable cv;
    bool sealed = false, failed = false, freed = false;
    bool sealing = false;          // a vb_shuffle_seal is running: a second caller waits for it instead of re-running
    u32 waiters = 0;               // threads blocked in wait_sealed: vb_shuffle_free drains them before deleting
    // export / import (world > 1)
    bool exported = false, imported = false;
    u64 *exp_keys = nullptr, *exp_vals = nullptr;
    // fused export (P2P): plan + scanned histogram + gathered input kept between export_counts and export_direct
    u32 *exp_hist = nullptr;
    u32 exp_parts = 0;
    u64 exp_rows_per_part = 0, exp_n = 0;
    const u64 *exp_rows = nullptr, *exp_k = nullptr, *exp_v = nullptr;
    std::vector<u64> exp_digit_start;
    bool exp_counted = false;
    const u64 *imp_keys = nullptr, *imp_vals = nullptr;
    u64 imp_n = 0;
    u64 *imp_own_k = nullptr, *imp_own_v = nullptr;   // receive buffers of vb_shuffle_exchange (freed with the inputs)
    std::vector<u64> sort_part_rows;                  // multi-rank sort: exact rows of every output partition this rank owns (0 elsewhere)
    vb_xstats xst{};
    // gathered input kept alive for the reduce side of group ops
    u64 *gath_keys = nullptr, *gath_vals = nullptr;
    // results
    u64 n_keys = 0, n_vals = 0;
    u64 *res_keys = nullptr, *res_comb = nullptr, *res_offs = nullptr, *res_vals = nullptr;
    std::vector<u64> bucket_off;   // n_reduce + 1 (key index)
    std::vector<u64> val_off;      // n_reduce + 1 (value index; group ops)
    void *dict = nullptr;          // group ops: key → slot table, kept for joins
    u32 dict_log_cap = 0;
    u32 *dense_of_slot = nullptr;
    std::map<std::pair<const vb_shuf *, u32>, JoinPlan> join_plans;
    std::map<std::pair<u64, u32>, CogroupPlan> cg_plans;   // by (right side's uid, reduce_id): kept from *_size to the fetch
    // COGROUP shuffles are grouped lazily: seal keeps the (owned) rows; the CSR is built by the first reduce call
    // (cogroup materialisation), or — if a join comes first — only for the keys that occur on BOTH sides.
    u64 uid = 0;                                   // process-unique id (cache key that survives pointer reuse)
    bool lazy = false;                             // sealed, rows in lz_*, not grouped yet
    u64 *lz_keys = nullptr, *lz_vals = nullptr;
    u64 lz_n = 0;
    std::vector<vb_shuf *> trash;                  // internal shuffles of a failed filtered join
    std::map<u64, std::pair<vb_shuf *, vb_shuf *>> filtered;   // by the right side's uid: internal (left, right) shuffles over the matching rows
    // stats
    vb_stats st{};
    std::vector<Timer> timers;
    double kms[K_N] = {0};
    u64 klaunch[K_N] = {0};
};

static bool is_reduce_op(int agg) { return agg == VB_AGG_SUM || agg == VB_AGG_MIN || agg == VB_AGG_MAX || agg == VB_AGG_COUNT; }
static bool is_group_op(int agg) { return agg == VB_AGG_GROUP || agg == VB_AGG_COGROUP; }

static int val_tx(const vb_shuf *s)
{
    if (s->agg != VB_AGG_MIN && s->agg != VB_AGG_MAX) return TX_NONE;
    return s->vdt == VB_I64 ? TX_I64 : s->vdt == VB_F64 ? TX_F64 : TX_NONE;
}
static int map_opk(const vb_shuf *s)
{
    switch (s->agg) {
    case VB_AGG_SUM: return s->vdt == VB_F64 ? OPK_ADD_F64 : OPK_ADD_U64;
    case VB_AGG_MIN: return OPK_MIN_U64;
    case VB_AGG_MAX: return OPK_MAX_U64;
    case VB_AGG_COUNT: return OPK_COUNT;
    default: return OPK_DICT;
    }
}
static int merge_opk(const vb_shuf *s) { return s->agg == VB_AGG_COUNT ? OPK_ADD_U64 : map_opk(s); }

// kernel launch bookkeeping (+ CUDA-event timing on the launching stream when profiling)
struct KLaunch {
    vb_shuf *s;
    int klass;
    u64 rows;
    cudaEvent_t a = nullptr, b = nullptr;
    bool pushed = false;
    ~KLaunch()
    {
        if (a && !pushed) { cudaEventDestroy(a); cudaEventDestroy(b); }
    }
    KLaunch(vb_shuf *s_, int klass_, u64 rows_ = 0) : s(s_), klass(klass_), rows(rows_)
    {
        if (s && s->ctx->profile) {
            cudaEventCreate(&a);
            cudaEventCreate(&b);
            cudaEventRecord(a, s->ctx->stream);
        }
    }
    int done(const char *what)
    {
        cudaError_t e = cudaGetLastError();
        if (a) {
            cudaEventRecord(b, s->ctx->stream);
            s->timers.push_back(Timer{a, b, klass, rows});
            pushed = true;
        }
        if (s && klass >= 0) {
            s->klaunch[klass]++;
            s->st.kernel_launches++;
        }
        if (e != cudaSuccess) return set_err(VB_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
        return VB_OK;
    }
};

static void resolve_timers(vb_shuf *s)
{
    if (s->timers.empty()) return;
    cudaStreamSynchronize(s->ctx->stream);
    for (auto &t : s->timers) {
        float ms = 0;
        if (cudaEventElapsedTime(&ms, t.a, t.b) == cudaSuccess) {
            if (t.klass >= 0) s->kms[t.klass] += ms;
            else if (t.klass == -1) s->st.map_ms += ms;
            else if (t.klass == -3) s->xst.exchange_ms += ms;
            else s->st.seal_ms += ms;
            int hot = is_reduce_op(s->agg) ? K_HASH_AGG : K_RP_SCATTER;
            if (t.klass == hot) {
                s->st.hot_kernel_ms += ms;
                s->st.hot_kernel_launches++;
                s->st.hot_kernel_rows += t.rows;
            }
        } else cudaGetLastError();
        cudaEventDestroy(t.a);
        cudaEventDestroy(t.b);
    }
    s->timers.clear();
}

static u32 ceil_log2_u64(u64 x)
{
    u32 l = 0;
    while ((1ull << l) < x && l < 63) ++l;
    return l;
}

// ---------------------------------------------------------------------------------------------
// hash table build (map-side combine / reduce-side merge / dictionary)
// ---------------------------------------------------------------------------------------------
struct AggInput {
    int in;          // IN_AOS / IN_SOA / IN_TABLE
    const u64 *a;
    const u64 *b;
    u64 n;           // rows (IN_TABLE: slots incl. the special one)
    int loc;         // VB_HOST or device
    u64 items = 0;   // IN_TABLE: upper bound on the occupied slots (n_inserted + 1); 0 = n
};

template <int IN, int OPK, int TX>
static int launch_hash_agg_t(vb_shuf *s, int klass, const u64 *a, const u64 *b, u64 n, void *tab, u32 log_cap,
                             TableCtl *ctl, u64 max_inserts, u32 *slot_out)
{
    vb_ctx *c = s->ctx;
    if constexpr (IN != IN_TABLE) {
        // bulk-staged (copy engine) variant: 16-byte aligned inputs of at least a few tiles per CTA
        static const bool no_bulk = getenv("VEGA_B200_NO_BULK") != nullptr;
        const bool aligned = (((uintptr_t)a | (uintptr_t)(b ? b : a)) & 15u) == 0;
        if (!no_bulk && aligned && n >= (u64)HB_TILE * 64) {
            auto kb = hash_agg_bulk_kernel<IN, OPK, TX>;
            constexpr bool has_v = (IN == IN_AOS) || (OPK != OPK_COUNT && OPK != OPK_DICT);
            const size_t smem = hb_smem_bytes(has_v);
            if (c->occ_cache.find((const void *)kb) == c->occ_cache.end())
                CU(cudaFuncSetAttribute(kb, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int occ = occupancy(c, kb, HB_THREADS, smem);
            u64 grid = std::min<u64>(n / HB_TILE, (u64)c->sm_count * occ);
            KLaunch kl(s, klass, n);
            if (klass == K_HASH_AGG) s->st.hot_kernel_variant = 1;
            kb<<<(unsigned)grid, HB_THREADS, smem, c->stream>>>(a, b, n, table_at(tab, log_cap), ctl, max_inserts, slot_out);
            return kl.done("hash_agg_bulk_kernel");
        }
    }
    auto kern = hash_agg_kernel<IN, OPK, TX>;
    int occ = occupancy(c, kern, HA_THREADS, 0);
    u64 tiles = (n + HA_TILE - 1) / HA_TILE;
    u64 grid = std::min<u64>(tiles, (u64)c->sm_count * occ);
    if (grid == 0) return VB_OK;
    KLaunch kl(s, klass, n);
    kern<<<(unsigned)grid, HA_THREADS, 0, c->stream>>>(a, b, n, table_at(tab, log_cap), ctl, max_inserts, slot_out);
    return kl.done("hash_agg_kernel");
}

template <int IN>
static int launch_hash_agg_in(vb_shuf *s, int klass, int opk, int tx, const u64 *a, const u64 *b, u64 n, void *tab,
                              u32 log_cap, TableCtl *ctl, u64 mi, u32 *so)
{
#define HA(O, T) return launch_hash_agg_t<IN, O, T>(s, klass, a, b, n, tab, log_cap, ctl, mi, so)
    switch (opk) {
    case OPK_ADD_U64: HA(OPK_ADD_U64, TX_NONE);
    case OPK_ADD_F64: HA(OPK_ADD_F64, TX_NONE);
    case OPK_COUNT: if constexpr (IN != IN_TABLE) { HA(OPK_COUNT, TX_NONE); } break;
    case OPK_DICT: if constexpr (IN != IN_TABLE) { HA(OPK_DICT, TX_NONE); } break;
    case OPK_MIN_U64:
        if (IN == IN_TABLE || tx == TX_NONE) HA(OPK_MIN_U64, TX_NONE);
        if (tx == TX_I64) HA(OPK_MIN_U64, (IN == IN_TABLE ? TX_NONE : TX_I64));
        HA(OPK_MIN_U64, (IN == IN_TABLE ? TX_NONE : TX_F64));
    case OPK_MAX_U64:
        if (IN == IN_TABLE || tx == TX_NONE) HA(OPK_MAX_U64, TX_NONE);
        if (tx == TX_I64) HA(OPK_MAX_U64, (IN == IN_TABLE ? TX_NONE : TX_I64));
        HA(OPK_MAX_U64, (IN == IN_TABLE ? TX_NONE : TX_F64));
    }
#undef HA
    return set_err(VB_ERR_UNSUPPORTED, "hash_agg: unsupported op %d for input mode %d", opk, IN);
}

static int launch_hash_agg(vb_shuf *s, int klass, int in, int opk, int tx, const u64 *a, const u64 *b, u64 n, void *tab,
                           u32 log_cap, TableCtl *ctl, u64 mi, u32 *so)
{
    switch (in) {
    case IN_AOS: return launch_hash_agg_in<IN_AOS>(s, klass, opk, tx, a, b, n, tab, log_cap, ctl, mi, so);
    case IN_SOA: return launch_hash_agg_in<IN_SOA>(s, klass, opk, tx, a, b, n, tab, log_cap, ctl, mi, so);
    case IN_TABLE: return launch_hash_agg_in<IN_TABLE>(s, klass, opk, tx, a, b, n, tab, log_cap, ctl, mi, so);
    }
    return set_err(VB_ERR_INVALID, "hash_agg: bad input mode %d", in);
}

constexpr u64 HOST_CHUNK_ROWS = 8ull << 20;    // host inputs stream through two 128 MiB staging halves (double-buffered)

// vega issues its map tasks concurrently from a tokio blocking pool (local_scheduler.rs:336-352).  A map call holds
// the context lock while it ENQUEUES copies and kernels, but waits for its own completion (table overflow flag,
// insert count) with the lock released, so the next task's H2D copies queue up behind this one's without a gap.
static thread_local std::unique_lock<std::mutex> *tl_ctx_lock = nullptr;

// D2H of `bytes` (<= 64) from `dev` at the current end of c->stream, waited for with the context unlocked.
static int fetch_status_unlocked(vb_ctx *c, const void *dev, void *out, size_t bytes)
{
    if (!tl_ctx_lock || c->pinned_slots.empty()) {          // not inside a map call: plain synchronous fetch
        CU(cudaMemcpyAsync(c->h_scratch, dev, bytes, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        memcpy(out, c->h_scratch, bytes);
        return VB_OK;
    }
    void *slot = c->pinned_slots.back();
    c->pinned_slots.pop_back();
    cudaEvent_t ev;
    CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    cudaError_t e = cudaMemcpyAsync(slot, dev, bytes, cudaMemcpyDeviceToHost, c->stream);
    if (e == cudaSuccess) e = cudaEventRecord(ev, c->stream);
    tl_ctx_lock->unlock();
    if (e == cudaSuccess) e = cudaEventSynchronize(ev);
    tl_ctx_lock->lock();
    cudaSetDevice(c->device);
    memcpy(out, slot, bytes);
    c->pinned_slots.push_back(slot);
    cudaEventDestroy(ev);
    if (e != cudaSuccess) { cudaGetLastError(); return set_err(VB_ERR_CUDA, "status fetch: %s", cudaGetErrorString(e)); }
    return VB_OK;
}
constexpr u32 MAX_LOG_CAP = 31;

static int launch_hash_agg(vb_shuf *s, int klass, int in, int opk, int tx, const u64 *a, const u64 *b, u64 n, void *tab,
                           u32 log_cap, TableCtl *ctl, u64 mi, u32 *so);

// Distinct-count estimate from a strided sample of up to 2^20 keys of the first device-resident
// input: insert the sample into a scratch dictionary, read the number of distinct keys d_s, and
// solve d_s = D (1 - exp(-s / D)) for D (keys assumed roughly equally frequent).  Returns 0 when
// there is nothing to sample; a sample that is ~all distinct only proves D >~ 25 s.
static int estimate_distinct(vb_shuf *s, const std::vector<AggInput> &inputs, u64 total, u64 *out)
{
    vb_ctx *c = s->ctx;
    *out = 0;
    const AggInput *src = nullptr;
    for (auto &in : inputs)
        if (in.loc != VB_HOST && in.n && (in.in == IN_AOS || in.in == IN_SOA)) { src = &in; break; }
    if (!src) return VB_OK;
    const u32 m = (u32)std::min<u64>(src->n, 1u << 20);
    const u64 stride = std::max<u64>(1, src->n / m);
    const u32 log_cap = 21;
    DevBuf keys(c), tab(c), ctl(c), slots(c);
    TRY(keys.alloc((size_t)m * 8));
    TRY(slots.alloc((size_t)m * 4));
    TRY(tab.alloc(table_bytes(log_cap)));
    TRY(ctl.alloc(sizeof(TableCtl)));
    CU(cudaMemsetAsync(ctl.p, 0, sizeof(TableCtl), c->stream));
    {
        KLaunch kl(s, K_MISC);
        table_init_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(table_at(tab.p, log_cap), 0);
        TRY(kl.done("table_init_kernel"));
    }
    {
        KLaunch kl(s, K_MISC);
        if (src->in == IN_AOS) sample_keys_kernel<IN_AOS><<<(m + 255) / 256, 256, 0, c->stream>>>(src->a, src->n, stride, keys.as<u64>(), m);
        else sample_keys_kernel<IN_SOA><<<(m + 255) / 256, 256, 0, c->stream>>>(src->a, src->n, stride, keys.as<u64>(), m);
        TRY(kl.done("sample_keys_kernel"));
    }
    TRY(launch_hash_agg(s, K_MISC, IN_SOA, OPK_DICT, TX_NONE, keys.as<u64>(), nullptr, m, tab.p, log_cap, ctl.as<TableCtl>(), ~0ull,
                        slots.as<u32>()));
    TableCtl *h = (TableCtl *)c->h_scratch;
    CU(cudaMemcpyAsync(h, ctl.p, sizeof(TableCtl), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    const double ds = (double)h->n_inserted + 1.0, sm = (double)m;
    double D;
    if (ds >= 0.98 * sm) {
        D = std::min<double>((double)total, 32.0 * sm);     // unresolved: at least ~25 s distinct keys
        if (src->n <= m) D = ds;                             // the sample was the whole input
    } else {
        double lo = ds, hi = 64.0 * sm;                      // d(D) = D (1 - exp(-s/D)) is increasing in D
        for (int it = 0; it < 60; ++it) {
            double mid = 0.5 * (lo + hi);
            if (mid * (1.0 - exp(-sm / mid)) < ds) lo = mid; else hi = mid;
        }
        D = hi;
    }
    *out = (u64)std::min<double>((double)total, D * 1.25 + 16.0);
    return VB_OK;
}

// First table size.  Load factor <= 0.4 while the table (16 B/slot) still fits comfortably in L2 (<= 64 MB),
// where a fuller 4-key bucket costs a second dependent probe (2.9 vs 2.2 ms per 2.5e8 rows at load 0.48 vs
// 0.24, profiles/r1_micro_v4_bucketized.log); <= 0.5 for bigger tables, which pay DRAM traffic instead.
static u32 choose_log_cap(u64 total, u64 hint_distinct, bool estimated, u32 max_log)
{
    u64 target = hint_distinct ? (hint_distinct * 5) / 2 : std::min<u64>(2 * std::max<u64>(total, 1), 1ull << 21);
    if (hint_distinct && target > (1ull << 22)) target = 2 * hint_distinct;
    // an estimate from a sample is a lower bound under skew: never start a large input below 2^21 slots (32 MB)
    if (estimated) target = std::max<u64>(target, 1ull << 21);
    return std::min(max_log, std::max<u32>(4, ceil_log2_u64(target)));
}

// Tables of 2^24 slots (256 MB) and more do not fit the 126 MB L2: every probe and every RED becomes a random
// DRAM access (57 ms per 1e9 rows at 1e7 keys, 86 ms at 1e8 — profiles/r1_cardinality_sweep_before_partitioning.jsonl).
// Such inputs are first radix-partitioned by the top bits of the slot hash (one stable 8-bit pass, ~10 ms per 1e9
// rows), so that consecutive tiles of hash_agg_kernel all probe the same <= 32 MB region of the table, which then
// stays L2-resident while it is being filled.  Reduce ops on device-resident rows only (the dictionary of group ops
// must keep row order, host inputs are PCIe-bound anyway).  VEGA_B200_NO_PARTITION=1 disables it.
struct PassPlan;
template <typename KeyT, bool HAS_VAL> static PassPlan plan_pass(vb_ctx *c, u64 n, int bits);
template <typename KeyT, bool HAS_VAL>
static int radix_pass(vb_shuf *s, const Loader &ld, const Digit &dg, u64 n, KeyT *out_keys, u64 *out_vals, u32 *d_hist, const PassPlan &plan,
                      u64 *csr = nullptr, bool *csr_done = nullptr);

constexpr u32 PARTITION_MIN_LOG_CAP = 24;

static bool want_partition(int in, int opk, u32 log_cap, u64 n)
{
    static const bool off = getenv("VEGA_B200_NO_PARTITION") != nullptr;
    return !off && opk != OPK_DICT && (in == IN_AOS || in == IN_SOA) && log_cap >= PARTITION_MIN_LOG_CAP && n >= (1ull << 22);
}

static int launch_hash_agg_partitioned(vb_shuf *s, int klass, int in, int opk, int tx, const u64 *a, const u64 *b, u64 n, void *tab,
                                       u32 log_cap, TableCtl *ctl, u64 mi);

// Feed every input into one fresh table; on overflow (abort flag) start again 4x larger.
// slot_out (OPK_DICT): one u32 per row over the concatenation of the inputs.
static int build_table(vb_shuf *s, int klass, const std::vector<AggInput> &inputs, int opk, int tx, u64 hint_distinct,
                       void **out_tab, u32 *out_log_cap, u64 *out_inserted, u32 *slot_out)
{
    vb_ctx *c = s->ctx;
    u64 total = 0;          // items that can each bring a new key (table inputs: occupied slots, not capacity)
    bool any_host = false;
    u64 max_host = 0;
    for (auto &in : inputs) {
        total += in.items ? std::min(in.items, in.n) : in.n;
        if (in.loc == VB_HOST) { any_host = true; max_host = std::max(max_host, in.n); }
    }
    if (slot_out && any_host) return set_err(VB_ERR_INVALID, "build_table: dictionary inputs must be on the device");
    // capacity never needs to exceed 2x the items; slot indices are 32-bit, so 2^31 slots is the ceiling — an input
    // with more than ~1.3e9 distinct keys fails with "overflow at maximum capacity", fewer distinct keys fit whatever the row count
    const u32 max_log = std::min<u32>(MAX_LOG_CAP, std::max<u32>(4, ceil_log2_u64(2 * std::max<u64>(total, 1))));
    bool estimated = false;
    if (!hint_distinct && total > (1ull << 20)) { TRY(estimate_distinct(s, inputs, total, &hint_distinct)); estimated = true; }
    u32 log_cap = choose_log_cap(total, hint_distinct, estimated, max_log);

    DevBuf ctl(c), stage_a(c), stage_b(c);
    TRY(ctl.alloc(sizeof(TableCtl)));
    const u64 stage_rows = std::min(max_host, HOST_CHUNK_ROWS);
    bool half_used[2] = {false, false};
    if (any_host) {
        TRY(stage_a.alloc(stage_rows * 16));   // per half: AoS rows, or SoA keys in the first 8 B/row / vals in the second
        TRY(stage_b.alloc(stage_rows * 16));
        CU(cudaEventRecord(c->ev_ready, c->stream));               // the pool hands the halves out in stream order
        CU(cudaStreamWaitEvent(c->copy_stream, c->ev_ready, 0));
    }
    TableCtl h_ctl_v;
    TableCtl *h_ctl = &h_ctl_v;
    for (;;) {
        const u64 cap = 1ull << log_cap;
        DevBuf tab(c);
        TRY(tab.alloc(table_bytes(log_cap)));
        {
            KLaunch kl(s, K_MISC);
            u64 blocks = std::min<u64>((cap + BUCKET + 255) / 256, (u64)c->sm_count * 8);
            table_init_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(table_at(tab.p, log_cap), op_identity(opk));
            TRY(kl.done("table_init_kernel"));
        }
        CU(cudaMemsetAsync(ctl.p, 0, sizeof(TableCtl), c->stream));
        const u64 max_inserts = (log_cap == max_log) ? ~0ull : (cap / 10) * 6;
        u64 row_base = 0;
        for (auto &in : inputs) {
            if (in.n == 0) continue;
            if (in.loc != VB_HOST && !slot_out && want_partition(in.in, opk, log_cap, in.n)) {
                TRY(launch_hash_agg_partitioned(s, klass, in.in, opk, tx, in.a, in.b, in.n, tab.p, log_cap, ctl.as<TableCtl>(), max_inserts));
            } else if (in.loc != VB_HOST) {
                TRY(launch_hash_agg(s, klass, in.in, opk, tx, in.a, in.b, in.n, tab.p, log_cap, ctl.as<TableCtl>(),
                                    max_inserts, slot_out ? slot_out + row_base : nullptr));
            } else {
                // double-buffered: the copy engine fills one half on the copy stream while hash_agg consumes the other
                const u64 chunk = std::min(in.n, stage_rows);
                u32 it = 0;
                for (u64 off = 0; off < in.n; off += chunk, ++it) {
                    const u64 m = std::min(chunk, in.n - off);
                    const u32 hb = it & 1u;
                    u64 *half = hb ? stage_b.as<u64>() : stage_a.as<u64>();
                    const u64 *da = half, *db = nullptr;
                    if (half_used[hb]) CU(cudaStreamWaitEvent(c->copy_stream, c->ev_kernel[hb], 0));   // its last reader is done
                    if (in.in == IN_AOS) {
                        CU(cudaMemcpyAsync(half, in.a + 2 * off, m * 16, cudaMemcpyHostToDevice, c->copy_stream));
                        s->st.h2d_bytes += m * 16;
                    } else {
                        CU(cudaMemcpyAsync(half, in.a + off, m * 8, cudaMemcpyHostToDevice, c->copy_stream));
                        s->st.h2d_bytes += m * 8;
                        if (in.b) {
                            db = half + chunk;
                            CU(cudaMemcpyAsync((void *)db, in.b + off, m * 8, cudaMemcpyHostToDevice, c->copy_stream));
                            s->st.h2d_bytes += m * 8;
                        }
                    }
                    CU(cudaEventRecord(c->ev_copied[hb], c->copy_stream));
                    CU(cudaStreamWaitEvent(c->stream, c->ev_copied[hb], 0));
                    TRY(launch_hash_agg(s, klass, in.in, opk, tx, da, db, m, tab.p, log_cap, ctl.as<TableCtl>(),
                                        max_inserts, nullptr));
                    CU(cudaEventRecord(c->ev_kernel[hb], c->stream));
                    half_used[hb] = true;
                }
            }
            row_base += in.n;
        }
        TRY(fetch_status_unlocked(c, ctl.p, h_ctl, sizeof(TableCtl)));     // waits with the context unlocked inside a map call
        if (!h_ctl->abort) {
            *out_tab = tab.release();
            *out_log_cap = log_cap;
            *out_inserted = h_ctl->n_inserted;
            s->st.table_slots = std::max<u64>(s->st.table_slots, cap);
            return VB_OK;
        }
        if (log_cap >= max_log) return set_err(VB_ERR_CUDA, "hash table overflow at maximum capacity 2^%u (internal error)", log_cap);
        log_cap = std::min(max_log, log_cap + 2);
        s->st.table_restarts++;
    }
}

// ---------------------------------------------------------------------------------------------
// radix pass host side
// ---------------------------------------------------------------------------------------------
struct PassPlan {
    u32 num_parts = 0;
    u64 rows_per_part = 0;
    u32 nb = RP_NB;     // bins of this pass
    size_t hist_bytes() const { return ((size_t)nb * num_parts + 1) * sizeof(u32); }
};

// (LDM, DGM, BITS) combinations the engine uses; anything else is a programming error.
// Multisplits (hash(K) % R, destination rank) use 8-bit digits, the LSD sorts 10-bit digits.
#define RP_COMBOS(X)                                                                                           \
    X(LD_SOA64, DG_BITS, RP_SORT_BITS) X(LD_AOS64, DG_BITS, RP_SORT_BITS)                                       \
    X(LD_KEY32_VAL_SOA, DG_BITS, RP_SORT_BITS) X(LD_KEY32_VAL_AOS, DG_BITS, RP_SORT_BITS)                       \
    X(LD_SOA64, DG_BUCKET, 8) X(LD_TABLE_KV, DG_BUCKET, 8) X(LD_TABLE_KI, DG_BUCKET, 8)                         \
    X(LD_SOA64, DG_DEST, 8) X(LD_AOS64, DG_DEST, 8) X(LD_TABLE_KV, DG_DEST, 8)                                 \
    X(LD_SOA64, DG_HASHTOP, 8) X(LD_AOS64, DG_HASHTOP, 8)

template <typename KeyT, int LDM> constexpr bool rp_key_ok()
{
    return (LDM == LD_KEY32_VAL_SOA || LDM == LD_KEY32_VAL_AOS) ? sizeof(KeyT) == 4 : sizeof(KeyT) == 8;
}

template <typename KeyT, bool HAS_VAL>
static const void *scatter_fn(int ldm, int dgm, int bits)
{
#define X(L, D, B) if (ldm == L && dgm == D && bits == B) { if constexpr (rp_key_ok<KeyT, L>()) return (const void *)rp_scatter_kernel<KeyT, HAS_VAL, L, D, B>; }
    RP_COMBOS(X)
#undef X
    return nullptr;
}

template <typename KeyT>
static const void *hist_fn(int ldm, int dgm, int bits)
{
#define X(L, D, B) if (ldm == L && dgm == D && bits == B) { if constexpr (rp_key_ok<KeyT, L>()) return (const void *)rp_hist_kernel<KeyT, L, D, B>; }
    RP_COMBOS(X)
#undef X
    return nullptr;
}

template <typename KeyT, bool HAS_VAL>
static size_t scatter_smem(int bits)
{
    return bits == 8 ? rp_scatter_smem<KeyT, HAS_VAL, 8>() : rp_scatter_smem<KeyT, HAS_VAL, RP_SORT_BITS>();
}

// The gather sweep (gsweep.cuh) is the scatter of the DG_BITS passes; VEGA_B200_NO_GSWEEP=1 falls back to rp_sweep_kernel<STATIC>.
static bool gsweep_enabled()
{
    static const bool on = getenv("VEGA_B200_NO_GSWEEP") == nullptr;
    return on;
}

template <typename KeyT, bool HAS_VAL>
static bool gsweep_lookup(int ldm, const void **kern, size_t *smem, u32 *tile, u32 *threads)
{
#define X(L)                                                                 \
    if (ldm == L) {                                                          \
        if constexpr (rp_key_ok<KeyT, L>() && (HAS_VAL || L == LD_SOA64)) { \
            *kern = (const void *)rp_gsweep_kernel<KeyT, HAS_VAL, L>;        \
            *smem = GsPlan<KeyT, HAS_VAL, L>::total;                         \
            *tile = (u32)GsPlan<KeyT, HAS_VAL, L>::T;                        \
            *threads = (u32)GsPlan<KeyT, HAS_VAL, L>::THREADS;               \
            return true;                                                     \
        }                                                                    \
    }
    X(LD_SOA64) X(LD_AOS64) X(LD_KEY32_VAL_SOA) X(LD_KEY32_VAL_AOS)
#undef X
    return false;
}

template <typename KeyT, bool HAS_VAL>
static PassPlan plan_pass(vb_ctx *c, u64 n, int bits)
{
    PassPlan p;
    p.nb = 1u << bits;
    if (n == 0) return p;
    // occupancy is the same for every loader/digit instantiation to within a CTA; use a representative one
    const void *kern = bits == 8 ? scatter_fn<KeyT, HAS_VAL>(LD_SOA64, DG_BUCKET, 8)
                                 : (sizeof(KeyT) == 4 ? scatter_fn<KeyT, HAS_VAL>(LD_KEY32_VAL_SOA, DG_BITS, bits)
                                                      : scatter_fn<KeyT, HAS_VAL>(LD_SOA64, DG_BITS, bits));
    size_t smem = scatter_smem<KeyT, HAS_VAL>(bits);
    int occ = 2;
    if (kern) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        occ = occupancy(c, kern, RPS_THREADS, smem);
    }
    if (bits == 8) occ = gsweep_enabled() ? GsPlan<KeyT, HAS_VAL, (sizeof(KeyT) == 4 ? LD_KEY32_VAL_SOA : LD_SOA64)>::CTAS
                                          : std::max(occ, sw_ctas<KeyT, HAS_VAL>());   // one part per resident CTA of the scatter that will run
    u64 tiles = (n + RP_TILE - 1) / RP_TILE;
    u64 parts = std::min<u64>(tiles, (u64)c->sm_count * occ);
    u64 tiles_per_part = (tiles + parts - 1) / parts;
    if (bits == 8 && tiles_per_part > 6) tiles_per_part = (tiles_per_part + 5) / 6 * 6;   // 24576-row units: a multiple of every sweep tile (3072 ... 8192 rows)
    p.rows_per_part = tiles_per_part * RP_TILE;
    p.num_parts = (u32)((n + p.rows_per_part - 1) / p.rows_per_part);
    return p;
}

// One stable pass: rows of `ld` (n of them) are written to out_keys/out_vals grouped by digit.
// d_hist (device, plan.hist_bytes()) afterwards holds the scanned histogram: d_hist[d*num_parts]
// is the output offset of digit d, d_hist[nb*num_parts] the number of valid rows.
template <typename KeyT>
static int radix_hist_scan(vb_shuf *s, const Loader &ld, const Digit &dg, u64 n, u32 *d_hist, const PassPlan &plan)
{
    vb_ctx *c = s->ctx;
    if (n == 0 || plan.num_parts == 0) return VB_OK;
    const int bits = plan.nb == 256 ? 8 : RP_SORT_BITS;
    const void *hk = hist_fn<KeyT>(ld.mode, dg.mode, bits);
    if (!hk) return set_err(VB_ERR_UNSUPPORTED, "radix pass: loader %d / digit %d / %d bits not instantiated", ld.mode, dg.mode, bits);
    const u64 tiles_per_part = plan.rows_per_part / RP_TILE;
    u32 split = (u32)std::max<u64>(1, std::min<u64>(tiles_per_part, ((u64)c->sm_count * 6 + plan.num_parts - 1) / plan.num_parts));
    CU(cudaMemsetAsync(d_hist, 0, plan.hist_bytes(), c->stream));
    u64 rows_per_part = plan.rows_per_part;
    u32 num_parts = plan.num_parts;
    Loader ldc = ld;
    Digit dgc = dg;
    {
        KLaunch kl(s, K_RP_HIST, n);
        void *args[] = {&ldc, &dgc, &n, &rows_per_part, &d_hist, &num_parts, &split};
        const size_t hsmem = rp_hist_smem(bits);
        CU(cudaFuncSetAttribute(hk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hsmem));
        CU(cudaLaunchKernel(hk, dim3(plan.num_parts * split), dim3(RP_THREADS), args, hsmem, c->stream));
        TRY(kl.done("rp_hist_kernel"));
    }
    {
        KLaunch kl(s, K_RP_SCAN);
        rp_scan_kernel<<<1, 1024, 0, c->stream>>>(d_hist, plan.nb * plan.num_parts);
        TRY(kl.done("rp_scan_kernel"));
    }
    return VB_OK;
}

template <typename KeyT, bool HAS_VAL>
static bool sweep_lookup(int ldm, int dgm, const void **kern, const void **hist, size_t *smem, const void **kern_static = nullptr);

template <typename KeyT, bool HAS_VAL>
static int radix_pass(vb_shuf *s, const Loader &ld, const Digit &dg, u64 n, KeyT *out_keys, u64 *out_vals, u32 *d_hist,
                      const PassPlan &plan, u64 *csr, bool *csr_done)
{
    vb_ctx *c = s->ctx;
    if (n == 0 || plan.num_parts == 0) return VB_OK;
    const int bits = plan.nb == 256 ? 8 : RP_SORT_BITS;
    const void *sk = scatter_fn<KeyT, HAS_VAL>(ld.mode, dg.mode, bits);
    if (!sk) return set_err(VB_ERR_UNSUPPORTED, "radix pass: loader %d / digit %d / %d bits not instantiated", ld.mode, dg.mode, bits);
    TRY((radix_hist_scan<KeyT>(s, ld, dg, n, d_hist, plan)));
    {   // LSD digit passes over row streams: the gather sweep (two 512-thread CTAs per SM, rows stay where the copy engine put them)
        const void *gk = nullptr;
        size_t gsm = 0;
        u32 GT = 0, gthreads = 0;
        if (gsweep_enabled() && bits == 8 && dg.mode == DG_BITS && n < SW_MAX_ROWS * 2 && plan.rows_per_part % 4096 == 0 &&
            gsweep_lookup<KeyT, HAS_VAL>(ld.mode, &gk, &gsm, &GT, &gthreads) && n >= 4ull * GT &&
            !(((uintptr_t)ld.keys & 15u) || (ld.vals && ((uintptr_t)ld.vals & 15u))) && !(HAS_VAL && ld.mode != LD_AOS64 && !ld.vals)) {
            if (c->occ_cache.find(gk) == c->occ_cache.end()) CU(cudaFuncSetAttribute(gk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm));
            (void)occupancy(c, gk, (int)gthreads, gsm);
            SweepArgs a{};
            a.keys = ld.keys; a.vals = ld.vals; a.n = n; a.n_tiles = 0;
            a.out_keys = out_keys; a.out_vals = out_vals;
            a.part_off = d_hist; a.num_parts = plan.num_parts; a.rows_per_part = plan.rows_per_part;
            if constexpr (sizeof(KeyT) == 4 && HAS_VAL) {
                // last pass of group_by_key's sort: value-run starts recorded by the scatter itself, ids not written (rp_gsweep_kernel<CSR>)
                static const bool no_csr = getenv("VEGA_B200_NO_CSR_FUSION") != nullptr;
                if (csr && !no_csr && ld.mode == LD_KEY32_VAL_SOA) {
                    const void *ck = (const void *)rp_gsweep_kernel<u32, true, LD_KEY32_VAL_SOA, true>;
                    if (c->occ_cache.find(ck) == c->occ_cache.end()) CU(cudaFuncSetAttribute(ck, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)gsm));
                    (void)occupancy(c, ck, (int)gthreads, gsm);
                    gk = ck;
                    a.csr = csr;
                    if (csr_done) *csr_done = true;
                }
            }
            static const u32 stagger = getenv("VEGA_B200_GS_STAGGER") ? (u32)atoi(getenv("VEGA_B200_GS_STAGGER")) : 0u;
            a.stagger_ns = stagger;
            Digit dgs = dg;
            KLaunch kl(s, K_RP_SCATTER, n);
            void *args[] = {&a, &dgs};
            CU(cudaLaunchKernel(gk, dim3(plan.num_parts), dim3(gthreads), args, gsm, c->stream));
            return kl.done("rp_gsweep_kernel");
        }
    }
    {   // row streams: the sweep tile pipeline fed by the per-part offsets (no look-back)
        static const bool off = getenv("VEGA_B200_NO_SWEEP_STATIC") != nullptr;
        const void *k0 = nullptr, *hk0 = nullptr, *kst = nullptr;
        size_t sm0 = 0;
        const u32 T = sw_tile<KeyT, HAS_VAL>();
        if (!off && bits == 8 && n < SW_MAX_ROWS * 2 && plan.rows_per_part % T == 0 && n >= 4ull * T &&
            sweep_lookup<KeyT, HAS_VAL>(ld.mode, dg.mode, &k0, &hk0, &sm0, &kst) &&
            !(((uintptr_t)ld.keys & 15u) || (ld.vals && ((uintptr_t)ld.vals & 15u))) && !(HAS_VAL && ld.mode != LD_AOS64 && !ld.vals)) {
            if (c->occ_cache.find(kst) == c->occ_cache.end()) CU(cudaFuncSetAttribute(kst, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm0));
            (void)occupancy(c, kst, sw_threads<KeyT, HAS_VAL>(), sm0);
            SweepArgs a{};
            a.keys = ld.keys; a.vals = ld.vals; a.n = n; a.n_tiles = (u32)((n + T - 1) / T);
            a.tile_counter = nullptr; a.state = nullptr; a.digit_base = nullptr;
            a.out_keys = out_keys; a.out_vals = out_vals;
            a.part_off = d_hist; a.num_parts = plan.num_parts; a.rows_per_part = plan.rows_per_part;
            Digit dgs = dg;
            KLaunch kl(s, K_RP_SCATTER, n);
            void *args[] = {&a, &dgs};
            CU(cudaLaunchKernel(kst, dim3(plan.num_parts), dim3(sw_threads<KeyT, HAS_VAL>()), args, sm0, c->stream));
            return kl.done("rp_sweep_kernel<STATIC>");
        }
    }
    const size_t smem = scatter_smem<KeyT, HAS_VAL>(bits);
    CU(cudaFuncSetAttribute(sk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    u64 rows_per_part = plan.rows_per_part;
    u32 num_parts = plan.num_parts;
    Loader ldc = ld;
    Digit dgc = dg;
    {
        KLaunch kl(s, K_RP_SCATTER, n);
        const u32 *ch = d_hist;
        RemoteDst rd{nullptr, nullptr, nullptr, 0};
        void *args[] = {&ldc, &dgc, &n, &rows_per_part, &ch, &num_parts, &out_keys, &out_vals, &rd};
        CU(cudaLaunchKernel(sk, dim3(plan.num_parts), dim3(RPS_THREADS), args, smem, c->stream));
        TRY(kl.done("rp_scatter_kernel"));
    }
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// sweep pass (sweep.cuh): one kernel per pass, decoupled look-back, copy-engine staged input
// ---------------------------------------------------------------------------------------------
#define SW_COMBOS_U64V(X) X(LD_SOA64, DG_BITS) X(LD_AOS64, DG_BITS) X(LD_SOA64, DG_DEST) X(LD_AOS64, DG_DEST) X(LD_SOA64, DG_HASHTOP) X(LD_AOS64, DG_HASHTOP) X(LD_SOA64, DG_BUCKET)
#define SW_COMBOS_U64K(X) X(LD_SOA64, DG_BITS)
#define SW_COMBOS_U32V(X) X(LD_KEY32_VAL_SOA, DG_BITS) X(LD_KEY32_VAL_AOS, DG_BITS)

template <typename KeyT, bool HAS_VAL>
static bool sweep_lookup(int ldm, int dgm, const void **kern, const void **hist, size_t *smem, const void **kern_static)
{
#define X(L, D)                                                                                   \
    if (ldm == L && dgm == D) {                                                                   \
        *kern = (const void *)rp_sweep_kernel<KeyT, HAS_VAL, L, D>;                               \
        if (kern_static) *kern_static = (const void *)rp_sweep_kernel<KeyT, HAS_VAL, L, D, true>; \
        *hist = (const void *)sw_hist_all_kernel<KeyT, L, D>;                                     \
        *smem = SwSmem<KeyT, HAS_VAL, L>::total;                                                  \
        return true;                                                                              \
    }
    if constexpr (sizeof(KeyT) == 8 && HAS_VAL) { SW_COMBOS_U64V(X) }
    if constexpr (sizeof(KeyT) == 8 && !HAS_VAL) { SW_COMBOS_U64K(X) }
    if constexpr (sizeof(KeyT) == 4 && HAS_VAL) { SW_COMBOS_U32V(X) }
#undef X
    return false;
}

// The one-kernel (look-back) pass is OPT-IN (VEGA_B200_SWEEP=1).  Measured on B200 (profiles/r2_sweep_bisection.jsonl,
// profiles/r2_ncu_sweep.txt): at ~22 tiles/us chip-wide the decoupled look-back needs ~40 predecessors per tile (three
// windows of 16 status words, each an L2 round trip spent behind a barrier) and costs ~3 ms per 1e9-row pass, which lands
// the pass at 10.9 ms — on par with histogram + scan + scatter (10.2 ms), not ahead of it.  The same tile pipeline WITHOUT
// the look-back (rp_sweep_kernel<STATIC>, fed by the per-part offsets) is the default scatter for row streams (radix_pass).
static bool sweep_enabled()
{
    static const bool on = getenv("VEGA_B200_SWEEP") != nullptr && getenv("VEGA_B200_NO_SWEEP") == nullptr;
    return on;
}

// rows of `ld` must be a plain row stream (every row valid) with 16-byte aligned column bases
template <typename KeyT, bool HAS_VAL>
static bool sweep_applicable(const Loader &ld, const Digit &dg, u64 n)
{
    const void *k, *h; size_t sm;
    if (!sweep_enabled() || n == 0 || n >= SW_MAX_ROWS) return false;
    if (!sweep_lookup<KeyT, HAS_VAL>(ld.mode, dg.mode, &k, &h, &sm)) return false;
    if (((uintptr_t)ld.keys & 15u) || (ld.vals && ((uintptr_t)ld.vals & 15u))) return false;
    if (HAS_VAL && ld.mode != LD_AOS64 && !ld.vals) return false;       // key-only rows in a (key, value) pass: the rp_* kernels fill zeros
    return true;
}

// Global histogram of `n_pos` digit positions in one read of the keys, scanned in place: d_bases[p][256].
template <typename KeyT, bool HAS_VAL>
static int sweep_hist(vb_shuf *s, const Loader &ld, const Digit &dg, u64 n, const HistAllArgs &ha, u32 *d_bases)
{
    vb_ctx *c = s->ctx;
    const void *kern, *hk; size_t smem;
    if (!sweep_lookup<KeyT, HAS_VAL>(ld.mode, dg.mode, &kern, &hk, &smem)) return set_err(VB_ERR_UNSUPPORTED, "sweep: loader %d / digit %d not instantiated", ld.mode, dg.mode);
    CU(cudaMemsetAsync(d_bases, 0, (size_t)ha.n_pos * SW_NB * 4, c->stream));
    Loader ldc = ld; Digit dgc = dg; HistAllArgs hac = ha;
    {
        KLaunch kl(s, K_RP_HIST, n);
        const unsigned grid = (unsigned)std::min<u64>((n + 2047) / 2048, (u64)c->sm_count * 4);
        void *args[] = {&ldc, &dgc, &n, &hac, &d_bases};
        CU(cudaLaunchKernel(hk, dim3(grid), dim3(512), args, 0, c->stream));
        TRY(kl.done("sw_hist_all_kernel"));
    }
    {
        KLaunch kl(s, K_RP_SCAN);
        sw_scan_bases_kernel<<<ha.n_pos, SW_NB, 0, c->stream>>>(d_bases, ha.n_pos);
        TRY(kl.done("sw_scan_bases_kernel"));
    }
    return VB_OK;
}

// One stable pass with the digit bases already on the device.  `scratch` (>= sweep_scratch_bytes) is reused across passes.
template <typename KeyT, bool HAS_VAL>
static size_t sweep_scratch_bytes(u64 n)
{
    const u64 tiles = (n + sw_tile<KeyT, HAS_VAL>() - 1) / sw_tile<KeyT, HAS_VAL>();
    return (size_t)(tiles * SW_NB + 4) * 4;
}

template <typename KeyT, bool HAS_VAL>
static int sweep_pass(vb_shuf *s, const Loader &ld, const Digit &dg, u64 n, KeyT *out_keys, u64 *out_vals, const u32 *d_base, u32 *scratch)
{
    vb_ctx *c = s->ctx;
    const void *kern, *hk; size_t smem;
    if (!sweep_lookup<KeyT, HAS_VAL>(ld.mode, dg.mode, &kern, &hk, &smem)) return set_err(VB_ERR_UNSUPPORTED, "sweep: loader %d / digit %d not instantiated", ld.mode, dg.mode);
    const u32 T = sw_tile<KeyT, HAS_VAL>();
    const u32 tiles = (u32)((n + T - 1) / T);
    CU(cudaMemsetAsync(scratch, 0, sweep_scratch_bytes<KeyT, HAS_VAL>(n), c->stream));
    if (c->occ_cache.find(kern) == c->occ_cache.end()) CU(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int occ = occupancy(c, kern, sw_threads<KeyT, HAS_VAL>(), smem);
    SweepArgs a;
    a.keys = ld.keys; a.vals = ld.vals; a.n = n; a.n_tiles = tiles;
    a.tile_counter = scratch; a.state = scratch + 4;
    a.digit_base = d_base; a.out_keys = out_keys; a.out_vals = out_vals;
    Digit dgc = dg;
    KLaunch kl(s, K_RP_SCATTER, n);
    const unsigned grid = (unsigned)std::min<u64>(tiles, (u64)c->sm_count * occ);
    void *args[] = {&a, &dgc};
    CU(cudaLaunchKernel(kern, dim3(grid), dim3(sw_threads<KeyT, HAS_VAL>()), args, smem, c->stream));
    return kl.done("rp_sweep_kernel");
}

static int launch_hash_agg_partitioned(vb_shuf *s, int klass, int in, int opk, int tx, const u64 *a, const u64 *b, u64 n, void *tab,
                                       u32 log_cap, TableCtl *ctl, u64 mi)
{
    vb_ctx *c = s->ctx;
    const u32 pbits = std::min<u32>(8, log_cap - 21);          // regions of <= 2^21 slots (32 MB) while 256 bins suffice
    DevBuf tk(c), tv(c), hist(c);
    TRY(tk.alloc(n * 8));
    TRY(tv.alloc(n * 8));
    PassPlan plan = plan_pass<u64, true>(c, n, 8);
    TRY(hist.alloc(plan.hist_bytes()));
    Loader ld = (in == IN_AOS) ? Loader{LD_AOS64, a, nullptr, 0} : Loader{LD_SOA64, a, b, 0};
    Digit dg{};
    dg.mode = DG_HASHTOP;
    dg.shift = 64 - pbits;
    dg.mask = (1u << pbits) - 1;
    if (sweep_applicable<u64, true>(ld, dg, n)) {
        DevBuf bases(c), scratch(c);
        TRY(bases.alloc(SW_NB * 4));
        TRY(scratch.alloc((sweep_scratch_bytes<u64, true>(n))));
        HistAllArgs ha{}; ha.n_pos = 1;
        TRY((sweep_hist<u64, true>(s, ld, dg, n, ha, bases.as<u32>())));
        TRY((sweep_pass<u64, true>(s, ld, dg, n, tk.as<u64>(), tv.as<u64>(), bases.as<u32>(), scratch.as<u32>())));
        return launch_hash_agg(s, klass, IN_SOA, opk, tx, tk.as<u64>(), tv.as<u64>(), n, tab, log_cap, ctl, mi, nullptr);
    }
    TRY((radix_pass<u64, true>(s, ld, dg, n, tk.as<u64>(), tv.as<u64>(), hist.as<u32>(), plan)));
    // stream-ordered frees: the buffers outlive the kernels queued on c->stream
    return launch_hash_agg(s, klass, IN_SOA, opk, tx, tk.as<u64>(), tv.as<u64>(), n, tab, log_cap, ctl, mi, nullptr);
}

// Copy the start offset of each of the first nb digits plus the total to the host: out[nb+1].
static int fetch_offsets(vb_ctx *c, const u32 *d_hist, const PassPlan &plan, u32 nb, u64 *out)
{
    u32 *h = (u32 *)c->h_scratch;
    CU(cudaMemcpy2DAsync(h, sizeof(u32), d_hist, (size_t)plan.num_parts * sizeof(u32), sizeof(u32), RP_NB,
                         cudaMemcpyDeviceToHost, c->stream));
    CU(cudaMemcpyAsync(h + RP_NB, d_hist + (size_t)RP_NB * plan.num_parts, sizeof(u32), cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    for (u32 d = 0; d < nb; ++d) out[d] = h[d];
    out[nb] = h[RP_NB];
    return VB_OK;
}

static Digit make_bucket_digit(const vb_shuf *s, int mode, u32 shift, u32 mask)
{
    Digit dg{};
    dg.mode = mode;
    dg.shift = shift;
    dg.mask = mask;
    dg.tx = TX_NONE;
    dg.key_width = s->key_width;
    dg.fm = make_fastmod(s->n_reduce);
    dg.fm_world = make_fastmod(s->world);
    return dg;
}

__global__ void bucket_hist_kernel(const u64 *__restrict__ keys, u64 n, Digit dg, u32 *__restrict__ cnt)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(&cnt[get_partition(keys[i], dg.key_width, dg.fm)], 1u);
}

// Unordered multisplit of a combined table's occupied slots (reduce ops only; <= 256 bins): see kernels.cuh.
static int multisplit_table_unordered(vb_shuf *s, const Table &t, int mode, u32 nbins, u64 *out_keys, u64 *out_vals, std::vector<u64> &bin_off)
{
    vb_ctx *c = s->ctx;
    bin_off.assign((size_t)nbins + 1, 0);
    const u64 cap = 1ull << t.log_cap;
    DevBuf cc(c);
    TRY(cc.alloc(2 * TS_MAX_BINS * 4));
    CU(cudaMemsetAsync(cc.p, 0, 2 * TS_MAX_BINS * 4, c->stream));
    u32 *counts = cc.as<u32>(), *cursors = cc.as<u32>() + TS_MAX_BINS;
    Digit dg = make_bucket_digit(s, mode, 0, 0xFFFFFFFFu);
    const unsigned grid = (unsigned)std::min<u64>((cap + TS_TILE) / TS_TILE, (u64)c->sm_count * 4);
    {
        KLaunch kl(s, K_RP_HIST, cap + 1);
        if (mode == DG_DEST) table_bin_count_kernel<DG_DEST><<<grid, TS_THREADS, 0, c->stream>>>(t.keys, cap, dg, counts);
        else table_bin_count_kernel<DG_BUCKET><<<grid, TS_THREADS, 0, c->stream>>>(t.keys, cap, dg, counts);
        TRY(kl.done("table_bin_count_kernel"));
    }
    {
        KLaunch kl(s, K_RP_SCATTER, cap + 1);
        if (mode == DG_DEST) table_bin_scatter_kernel<DG_DEST><<<grid, TS_THREADS, 0, c->stream>>>(t.keys, t.accs, cap, dg, counts, cursors, out_keys, out_vals);
        else table_bin_scatter_kernel<DG_BUCKET><<<grid, TS_THREADS, 0, c->stream>>>(t.keys, t.accs, cap, dg, counts, cursors, out_keys, out_vals);
        TRY(kl.done("table_bin_scatter_kernel"));
    }
    u32 *h = (u32 *)c->h_scratch;
    CU(cudaMemcpyAsync(h, counts, TS_MAX_BINS * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    u64 run = 0;
    for (u32 d = 0; d < nbins; ++d) { bin_off[d] = run; run += h[d]; }
    bin_off[nbins] = run;
    return VB_OK;
}

// Stable multisplit of `n` loader rows by reduce partition (DG_BUCKET, nbins = n_reduce) or by
// owning rank (DG_DEST, nbins = world).  Invalid rows (empty table slots) are dropped.
// out_keys/out_vals must hold `max_valid` rows.  bin_off[nbins+1] (host) gets the offsets.
static int multisplit(vb_shuf *s, const Loader &ld, u64 n, int mode, u32 nbins, u64 max_valid, u64 *out_keys, u64 *out_vals,
                      std::vector<u64> &bin_off)
{
    vb_ctx *c = s->ctx;
    bin_off.assign((size_t)nbins + 1, 0);
    if (n == 0) return VB_OK;
    if (nbins <= RP_NB) {
        Digit dg = make_bucket_digit(s, mode, 0, 0xFFFFFFFFu);
        if (sweep_applicable<u64, true>(ld, dg, n)) {          // row streams: one look-back pass + one histogram read
            DevBuf bases(c), scratch(c);
            TRY(bases.alloc(SW_NB * 4));
            TRY(scratch.alloc((sweep_scratch_bytes<u64, true>(n))));
            HistAllArgs ha{}; ha.n_pos = 1;
            TRY((sweep_hist<u64, true>(s, ld, dg, n, ha, bases.as<u32>())));
            TRY((sweep_pass<u64, true>(s, ld, dg, n, out_keys, out_vals, bases.as<u32>(), scratch.as<u32>())));
            u32 *h = (u32 *)c->h_scratch;
            CU(cudaMemcpyAsync(h, bases.p, SW_NB * 4, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            for (u32 d = 0; d < nbins; ++d) bin_off[d] = h[d];
            bin_off[nbins] = n;
            return VB_OK;
        }
    }
    PassPlan plan = plan_pass<u64, true>(c, n, 8);
    DevBuf hist(c);
    TRY(hist.alloc(plan.hist_bytes()));
    if (nbins <= RP_NB) {
        Digit dg = make_bucket_digit(s, mode, 0, 0xFFFFFFFFu);
        TRY((radix_pass<u64, true>(s, ld, dg, n, out_keys, out_vals, hist.as<u32>(), plan)));
        TRY(fetch_offsets(c, hist.as<u32>(), plan, nbins, bin_off.data()));
        return VB_OK;
    }
    if (mode != DG_BUCKET || nbins > 65536) return set_err(VB_ERR_UNSUPPORTED, "more than 65536 reduce partitions / 256 ranks");
    // two LSD passes over the 16-bit bucket id
    DevBuf tk(c), tv(c);
    TRY(tk.alloc(max_valid * 8));
    TRY(tv.alloc(max_valid * 8));
    Digit d0 = make_bucket_digit(s, DG_BUCKET, 0, 0xFF);
    TRY((radix_pass<u64, true>(s, ld, d0, n, tk.as<u64>(), tv.as<u64>(), hist.as<u32>(), plan)));
    std::vector<u64> tmp(RP_NB + 1);
    TRY(fetch_offsets(c, hist.as<u32>(), plan, RP_NB, tmp.data()));
    const u64 nv = tmp[RP_NB];
    if (nv == 0) return VB_OK;
    PassPlan plan2 = plan_pass<u64, true>(c, nv, 8);
    DevBuf hist2(c);
    TRY(hist2.alloc(plan2.hist_bytes()));
    Loader l2{LD_SOA64, tk.p, tv.p, 0};
    Digit d1 = make_bucket_digit(s, DG_BUCKET, 8, 0xFF);
    TRY((radix_pass<u64, true>(s, l2, d1, nv, out_keys, out_vals, hist2.as<u32>(), plan2)));
    DevBuf cnt(c);
    TRY(cnt.alloc((size_t)nbins * 4));
    CU(cudaMemsetAsync(cnt.p, 0, (size_t)nbins * 4, c->stream));
    {
        KLaunch kl(s, K_MISC);
        bucket_hist_kernel<<<(unsigned)((nv + 255) / 256), 256, 0, c->stream>>>(out_keys, nv, d0, cnt.as<u32>());
        TRY(kl.done("bucket_hist_kernel"));
    }
    std::vector<u32> hc(nbins);
    CU(cudaMemcpyAsync(hc.data(), cnt.p, (size_t)nbins * 4, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    u64 run = 0;
    for (u32 b = 0; b < nbins; ++b) { bin_off[b] = run; run += hc[b]; }
    bin_off[nbins] = run;
    return VB_OK;
}

// LSD radix sort of (u32 id, u64 val) pairs over `bits` low bits.  ids_a is overwritten.
// The first pass reads values through `first` (ids come from ids_a).  Results: *out_ids, *out_vals
// (owned by the caller afterwards).
static int sort_id_pairs(vb_shuf *s, u32 *ids_a, const Loader &first, u64 n, u32 bits, u32 **out_ids, u64 **out_vals, const u32 *xlat = nullptr,
                         u64 *csr = nullptr, bool *csr_done = nullptr)
{
    vb_ctx *c = s->ctx;
    const u32 passes = std::max<u32>(1, (bits + RP_SORT_BITS - 1) / RP_SORT_BITS);
    if (xlat) {                               // slot ids -> dense ids, in place
        KLaunch kl(s, K_MISC);
        u64 blocks = std::min<u64>((n + 255) / 256, (u64)c->sm_count * 8);
        translate_ids_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(ids_a, n, xlat);
        TRY(kl.done("translate_ids_kernel"));
    }
    {
        Loader probe = first;
        probe.keys = ids_a;
        Digit dgp{};
        dgp.mode = DG_BITS;
        if (sweep_applicable<u32, true>(probe, dgp, n) && RP_SORT_BITS == 8) {
            // sweep path: ONE histogram read for all digit positions, then one look-back kernel per pass
            DevBuf bases(c), scratch(c), ids_b(c), vals_a(c), vals_b(c);
            TRY(bases.alloc((size_t)passes * SW_NB * 4));
            TRY(scratch.alloc((sweep_scratch_bytes<u32, true>(n))));
            TRY(ids_b.alloc(n * 4));
            TRY(vals_b.alloc(n * 8));
            if (passes >= 2) TRY(vals_a.alloc(n * 8));
            HistAllArgs ha{};
            ha.n_pos = passes;
            for (u32 p = 0; p < passes; ++p) ha.shifts[p] = 8 * p;
            Loader lk{LD_KEY32_VAL_SOA, ids_a, nullptr, 0};
            TRY((sweep_hist<u32, true>(s, lk, dgp, n, ha, bases.as<u32>())));
            u32 *src_ids = ids_a, *dst_ids = ids_b.as<u32>();
            u64 *src_vals = nullptr, *dst_vals = vals_b.as<u64>();
            for (u32 p = 0; p < passes; ++p) {
                Loader ld = first;
                if (p == 0) ld.keys = src_ids;
                else ld = Loader{LD_KEY32_VAL_SOA, src_ids, src_vals, 0};
                Digit dg{};
                dg.mode = DG_BITS; dg.shift = 8 * p; dg.mask = 0xFF; dg.tx = TX_NONE;
                TRY((sweep_pass<u32, true>(s, ld, dg, n, dst_ids, dst_vals, bases.as<u32>() + (size_t)p * SW_NB, scratch.as<u32>())));
                std::swap(src_ids, dst_ids);
                u64 *nv = (src_vals == nullptr) ? vals_a.as<u64>() : src_vals;
                src_vals = dst_vals;
                dst_vals = nv;
            }
            *out_ids = src_ids;
            *out_vals = src_vals;
            if (src_ids == ids_b.as<u32>()) ids_b.release();
            if (src_vals == vals_b.as<u64>()) vals_b.release(); else vals_a.release();
            return VB_OK;
        }
    }
    PassPlan plan = plan_pass<u32, true>(c, n, RP_SORT_BITS);
    DevBuf hist(c), ids_b(c), vals_a(c), vals_b(c);
    TRY(hist.alloc(plan.hist_bytes()));
    TRY(ids_b.alloc(n * 4));
    TRY(vals_b.alloc(n * 8));
    if (passes >= 2) TRY(vals_a.alloc(n * 8));
    u32 *src_ids = ids_a, *dst_ids = ids_b.as<u32>();
    u64 *src_vals = nullptr, *dst_vals = vals_b.as<u64>();
    for (u32 p = 0; p < passes; ++p) {
        Loader ld = first;
        if (p == 0) ld.keys = src_ids;
        else ld = Loader{LD_KEY32_VAL_SOA, src_ids, src_vals, 0};
        Digit dg{};
        dg.mode = DG_BITS;
        dg.shift = RP_SORT_BITS * p;
        dg.mask = (1u << RP_SORT_BITS) - 1;
        dg.tx = TX_NONE;
        const bool last = (p + 1 == passes);
        TRY((radix_pass<u32, true>(s, ld, dg, n, dst_ids, dst_vals, hist.as<u32>(), plan, last ? csr : nullptr, last ? csr_done : nullptr)));
        std::swap(src_ids, dst_ids);
        u64 *nv = (src_vals == nullptr) ? vals_a.as<u64>() : src_vals;
        src_vals = dst_vals;
        dst_vals = nv;
    }
    // results are in src_ids / src_vals
    *out_ids = src_ids;
    *out_vals = src_vals;
    if (src_ids == ids_b.as<u32>()) ids_b.release();          // ids_a stays with the caller either way
    if (src_vals == vals_b.as<u64>()) vals_b.release(); else vals_a.release();
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// shuffle lifecycle
// ---------------------------------------------------------------------------------------------
extern "C" int32_t vb_shuffle_create(vb_ctx *c, uint64_t shuffle_id, uint32_t n_map, uint32_t n_reduce, int32_t kdt,
                                     int32_t vdt, int32_t agg, int32_t part, vb_shuf **out)
{
    if (!c || !out) return set_err(VB_ERR_INVALID, "vb_shuffle_create: NULL argument");
    *out = nullptr;
    if (n_reduce < 1) return set_err(VB_ERR_INVALID, "vb_shuffle_create: n_reduce must be >= 1");
    if (kdt < VB_U64 || kdt > VB_F64 || vdt < VB_U64 || vdt > VB_F64) return set_err(VB_ERR_INVALID, "bad dtype");
    if (agg < VB_AGG_GROUP || agg > VB_AGG_SORT) return set_err(VB_ERR_INVALID, "bad agg %d", agg);
    if (agg != VB_AGG_SORT && kdt == VB_F64) return set_err(VB_ERR_UNSUPPORTED, "f64 keys are not hashable (Rust f64 is not Hash)");
    if ((agg == VB_AGG_SORT) != (part == VB_PART_RANGE)) return set_err(VB_ERR_INVALID, "VB_PART_RANGE goes with VB_AGG_SORT only");
    if (n_reduce > 65536) return set_err(VB_ERR_UNSUPPORTED, "more than 65536 reduce partitions");
    vb_shuf *s = new vb_shuf();
    static std::atomic<u64> next_uid{1};
    s->uid = next_uid.fetch_add(1);
    s->ctx = c;
    s->id = shuffle_id;
    s->n_map = n_map;
    s->n_reduce = n_reduce;
    s->kdt = kdt;
    s->vdt = vdt;
    s->agg = agg;
    s->part = part;
    s->maps.resize(n_map);
    *out = s;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_set_key_width(vb_shuf *s, uint32_t bytes)
{
    if (!s || (bytes != 4 && bytes != 8)) return set_err(VB_ERR_INVALID, "key width must be 4 or 8");
    s->key_width = bytes;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_set_hint(vb_shuf *s, uint64_t d)
{
    if (!s) return set_err(VB_ERR_INVALID, "NULL shuffle");
    s->hint = d;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_set_dist(vb_shuf *s, uint32_t rank, uint32_t world)
{
    if (!s || world < 1 || rank >= world || world > 256) return set_err(VB_ERR_INVALID, "bad rank/world");
    s->rank = rank;
    s->world = world;
    return VB_OK;
}

static void free_map(vb_shuf *s, MapOut &m)
{
    vb_ctx *c = s->ctx;
    if (m.table) dev_free(c, m.table);
    if (m.owned) { dev_free(c, m.rows); dev_free(c, m.keys); dev_free(c, m.vals); }
    m = MapOut();
}

static int shuffle_map(vb_shuf *s, u32 map_id, const u64 *rows, const u64 *keys, const u64 *vals, u64 n, int loc, bool combined = false)
{
    if (!s) return set_err(VB_ERR_INVALID, "NULL shuffle");
    if (map_id >= s->n_map) return set_err(VB_ERR_INVALID, "map_id %u >= n_map %u", map_id, s->n_map);
    if (loc < VB_HOST || loc > VB_DEVICE_BORROWED) return set_err(VB_ERR_INVALID, "bad src_loc %d", loc);
    if (n && !rows && !keys) return set_err(VB_ERR_INVALID, "NULL input with n_rows > 0");
    if (n >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "map partition of %llu rows", (unsigned long long)n);
    vb_ctx *c = s->ctx;
    {
        std::lock_guard<std::mutex> g(s->mu);
        if (s->sealed || s->exported || s->freed) return set_err(VB_ERR_STATE, "shuffle %llu: map after seal/export", (unsigned long long)s->id);
    }
    std::unique_lock<std::mutex> lk(c->mu);
    struct TlGuard { TlGuard(std::unique_lock<std::mutex> *l) { tl_ctx_lock = l; } ~TlGuard() { tl_ctx_lock = nullptr; } } tlg(&lk);
    CU(cudaSetDevice(c->device));
    KLaunch call(s, -1);
    MapOut &m = s->maps[map_id];
    if (m.present) {                                                // stage resubmission: overwrite
        if (m.in_shared) s->sh_dirty = true;                        // its rows are already in the shared table: rebuild at seal
        s->st.rows_in -= m.n_rows;
        free_map(s, m);
    }
    m.n_rows = n;
    if (is_reduce_op(s->agg) && loc == VB_DEVICE_BORROWED && !combined) {
        if (!rows && !vals && s->agg != VB_AGG_COUNT && n) return set_err(VB_ERR_INVALID, "values required for this aggregator");
        std::vector<AggInput> in(1);
        in[0] = AggInput{rows ? IN_AOS : IN_SOA, rows ? rows : keys, vals, n, VB_DEVICE};
        if (!s->sh_tab && !s->sh_dirty && n) {       // first borrowed map task: size and create the shared table
            u64 hint = s->hint;
            bool estimated = false;
            const u64 total_guess = n * std::max<u64>(1, s->n_map / std::max<u32>(1, s->world));
            if (!hint && n > (1ull << 20)) { TRY(estimate_distinct(s, in, total_guess, &hint)); estimated = true; }
            const u32 max_log = std::min<u32>(MAX_LOG_CAP, std::max<u32>(4, ceil_log2_u64(2 * std::max<u64>(total_guess, 1))));
            s->sh_log_cap = choose_log_cap(total_guess, hint, estimated, max_log);
            DevBuf tab(c), ctl(c);
            TRY(tab.alloc(table_bytes(s->sh_log_cap)));
            TRY(ctl.alloc(sizeof(TableCtl)));
            CU(cudaMemsetAsync(ctl.p, 0, sizeof(TableCtl), c->stream));
            {
                KLaunch kl(s, K_MISC);
                const u64 cap = 1ull << s->sh_log_cap;
                u64 blocks = std::min<u64>((cap + BUCKET + 255) / 256, (u64)c->sm_count * 8);
                table_init_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(table_at(tab.p, s->sh_log_cap), op_identity(map_opk(s)));
                TRY(kl.done("table_init_kernel"));
            }
            s->sh_max_inserts = (s->sh_log_cap >= max_log) ? ~0ull : ((1ull << s->sh_log_cap) / 10) * 6;
            s->sh_tab = tab.release();
            s->sh_ctl = (TableCtl *)ctl.release();
            s->st.table_slots = std::max<u64>(s->st.table_slots, 1ull << s->sh_log_cap);
        }
        if (s->sh_tab && !s->sh_dirty && n) {         // asynchronous: checked at seal
            if (want_partition(in[0].in, map_opk(s), s->sh_log_cap, n))
                TRY(launch_hash_agg_partitioned(s, K_HASH_AGG, in[0].in, map_opk(s), val_tx(s), in[0].a, in[0].b, n, s->sh_tab, s->sh_log_cap,
                                                s->sh_ctl, s->sh_max_inserts));
            else
                TRY(launch_hash_agg(s, K_HASH_AGG, in[0].in, map_opk(s), val_tx(s), in[0].a, in[0].b, n, s->sh_tab, s->sh_log_cap, s->sh_ctl,
                                    s->sh_max_inserts, nullptr));
        }
        m.rows = rows; m.keys = keys; m.vals = vals; m.owned = false; m.in_shared = true;
    } else if (is_reduce_op(s->agg)) {
        if (!rows && !vals && s->agg != VB_AGG_COUNT && n) return set_err(VB_ERR_INVALID, "values required for this aggregator");
        std::vector<AggInput> in(1);
        in[0] = AggInput{rows ? IN_AOS : IN_SOA, rows ? rows : keys, vals, n, loc == VB_HOST ? VB_HOST : VB_DEVICE};
        const u64 hint = s->hint ? s->hint : (s->learned_distinct ? s->learned_distinct + s->learned_distinct / 4 : 0);
        // a map-side-combined bucket carries combiners, merged with merge_combiners (partial counts are summed)
        TRY(build_table(s, K_HASH_AGG, in, combined ? merge_opk(s) : map_opk(s), val_tx(s), hint, &m.table, &m.log_cap, &m.n_inserted, nullptr));
        s->learned_distinct = std::max<u64>(m.n_inserted, 1);
    } else if (n) {
        if (loc == VB_DEVICE_BORROWED) {
            m.rows = rows; m.keys = keys; m.vals = vals; m.owned = false;
        } else {
            const cudaMemcpyKind kind = loc == VB_HOST ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
            DevBuf a(c), b(c);
            // the copies run on the copy stream (ordered after the pool's hand-out), so a concurrent map task's kernels
            // on c->stream are not held up by this task's PCIe transfer
            if (rows) TRY(a.alloc(n * 16));
            else { TRY(a.alloc(n * 8)); if (vals) TRY(b.alloc(n * 8)); }
            cudaEvent_t ev_in, ev_done;
            CU(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
            CU(cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming));
            CU(cudaEventRecord(ev_in, c->stream));
            CU(cudaStreamWaitEvent(c->copy_stream, ev_in, 0));
            if (rows) {
                CU(cudaMemcpyAsync(a.p, rows, n * 16, kind, c->copy_stream));
                if (loc == VB_HOST) s->st.h2d_bytes += n * 16;
            } else {
                CU(cudaMemcpyAsync(a.p, keys, n * 8, kind, c->copy_stream));
                if (loc == VB_HOST) s->st.h2d_bytes += n * 8;
                if (vals) {
                    CU(cudaMemcpyAsync(b.p, vals, n * 8, kind, c->copy_stream));
                    if (loc == VB_HOST) s->st.h2d_bytes += n * 8;
                }
            }
            CU(cudaEventRecord(ev_done, c->copy_stream));
            CU(cudaStreamWaitEvent(c->stream, ev_done, 0));      // later work on c->stream sees the rows
            lk.unlock();                                         // the caller may reuse its buffer on return: wait, unlocked
            cudaError_t ce = cudaEventSynchronize(ev_done);
            lk.lock();
            cudaSetDevice(c->device);
            cudaEventDestroy(ev_in); cudaEventDestroy(ev_done);
            if (ce != cudaSuccess) { cudaGetLastError(); return set_err(VB_ERR_CUDA, "input copy: %s", cudaGetErrorString(ce)); }
            if (rows) m.rows = (const u64 *)a.release();
            else { m.keys = (const u64 *)a.release(); m.vals = vals ? (const u64 *)b.release() : nullptr; }
            m.owned = true;
        }
    }
    m.present = true;
    s->st.rows_in += n;
    TRY(call.done("map"));
    return VB_OK;
}

extern "C" int32_t vb_shuffle_map_aos(vb_shuf *s, uint32_t map_id, const void *rows, uint64_t n, int32_t loc)
{
    return shuffle_map(s, map_id, (const u64 *)rows, nullptr, nullptr, n, loc);
}
extern "C" int32_t vb_shuffle_map_soa(vb_shuf *s, uint32_t map_id, const void *keys, const void *vals, uint64_t n, int32_t loc)
{
    return shuffle_map(s, map_id, nullptr, (const u64 *)keys, (const u64 *)vals, n, loc);
}

// ---------------------------------------------------------------------------------------------
// reduce side
// ---------------------------------------------------------------------------------------------
// Concatenate the rows of all present map partitions in map-id order.  Zero-copy when they are
// one AoS run (adjacent in memory) or a single partition; otherwise SoA copies owned by s.
struct Gathered {
    const u64 *rows = nullptr, *keys = nullptr, *vals = nullptr;
    u64 n = 0;
};

static int gather_maps(vb_shuf *s, Gathered *g)
{
    vb_ctx *c = s->ctx;
    u64 n = 0;
    std::vector<MapOut *> segs;
    for (auto &m : s->maps)
        if (m.present && m.n_rows) { segs.push_back(&m); n += m.n_rows; }
    g->n = n;
    if (n == 0) return VB_OK;
    if (n >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "shuffle of %llu rows on one device", (unsigned long long)n);
    bool contiguous = true;
    for (size_t i = 0; i < segs.size(); ++i) {
        if (!segs[i]->rows) { contiguous = false; break; }
        if (i && segs[i - 1]->rows + 2 * segs[i - 1]->n_rows != segs[i]->rows) { contiguous = false; break; }
    }
    if (contiguous) { g->rows = segs[0]->rows; return VB_OK; }
    if (segs.size() == 1) { g->keys = segs[0]->keys; g->vals = segs[0]->vals; return VB_OK; }
    bool any_vals = false;
    for (auto *m : segs) any_vals |= (m->rows != nullptr) || (m->vals != nullptr);
    DevBuf k(c), v(c);
    TRY(k.alloc(n * 8));
    if (any_vals) TRY(v.alloc(n * 8));
    u64 off = 0;
    for (auto *m : segs) {
        if (m->rows) {
            KLaunch kl(s, K_MISC);
            u64 blocks = std::min<u64>((m->n_rows + 255) / 256, (u64)c->sm_count * 8);
            aos_to_soa_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(m->rows, m->n_rows, k.as<u64>() + off, v.as<u64>() + off);
            TRY(kl.done("aos_to_soa_kernel"));
        } else {
            CU(cudaMemcpyAsync(k.as<u64>() + off, m->keys, m->n_rows * 8, cudaMemcpyDeviceToDevice, c->stream));
            if (any_vals) {
                if (m->vals) CU(cudaMemcpyAsync(v.as<u64>() + off, m->vals, m->n_rows * 8, cudaMemcpyDeviceToDevice, c->stream));
                else CU(cudaMemsetAsync(v.as<u64>() + off, 0, m->n_rows * 8, c->stream));
            }
        }
        off += m->n_rows;
    }
    s->gath_keys = (u64 *)k.release();
    s->gath_vals = any_vals ? (u64 *)v.release() : nullptr;
    g->keys = s->gath_keys;
    g->vals = s->gath_vals;
    for (auto &m : s->maps) if (m.present && m.owned) { dev_free(c, m.rows); dev_free(c, m.keys); dev_free(c, m.vals); m.rows = m.keys = m.vals = nullptr; m.owned = false; }
    return VB_OK;
}

__global__ void gather_u64_kernel(const u64 *__restrict__ src, const u64 *__restrict__ idx, u32 n, u64 *__restrict__ out)
{
    u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[idx[i]];
}

__global__ void rebase_kernel(const u64 *__restrict__ src, u64 n, u64 base, u64 *__restrict__ out)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = src[i] - base;
}

// group_by_key / cogroup reduce side over n rows (AoS `rows`, or SoA keys/vals).
static int seal_group(vb_shuf *s, const Gathered &g)
{
    vb_ctx *c = s->ctx;
    const u32 R = s->n_reduce;
    s->bucket_off.assign((size_t)R + 1, 0);
    s->val_off.assign((size_t)R + 1, 0);
    const u64 n = g.n;
    if (n == 0) return VB_OK;
    // 1. dictionary: key → slot, slot per row
    DevBuf ids(c);
    TRY(ids.alloc(n * 4));
    std::vector<AggInput> in(1);
    in[0] = AggInput{g.rows ? IN_AOS : IN_SOA, g.rows ? g.rows : g.keys, nullptr, n, VB_DEVICE};
    u64 n_ins = 0;
    TRY(build_table(s, K_DICT, in, OPK_DICT, TX_NONE, s->hint, &s->dict, &s->dict_log_cap, &n_ins, ids.as<u32>()));
    const u64 cap = 1ull << s->dict_log_cap;
    // 2. distinct keys grouped by reduce partition (stable by slot)
    const u64 max_d = n_ins + 1;
    DevBuf ckeys(c), cslot(c);
    TRY(ckeys.alloc(max_d * 8));
    TRY(cslot.alloc(max_d * 8));
    const Table dt = table_at(s->dict, s->dict_log_cap);
    Loader lt{LD_TABLE_KI, dt.keys, nullptr, cap};
    TRY(multisplit(s, lt, cap + 1, DG_BUCKET, R, max_d, ckeys.as<u64>(), cslot.as<u64>(), s->bucket_off));
    const u64 D = s->bucket_off[R];
    // 3. slot → dense id (bucket-major)
    DevBuf dense(c);
    TRY(dense.alloc((cap + 1) * 4));
    {
        KLaunch kl(s, K_MISC);
        scatter_dense_kernel<<<(unsigned)((D + 255) / 256), 256, 0, c->stream>>>(cslot.as<u64>(), (u32)D, dense.as<u32>());
        TRY(kl.done("scatter_dense_kernel"));
    }
    cslot.reset();
    // 4. ids[i] = dense_of_slot[slot_of_row[i]]: first thing sort_id_pairs does (translate_ids_kernel)
    // 5. stable LSD sort of (id, value) — the reduce partition is the high part of the dense id
    Loader first = g.rows ? Loader{LD_KEY32_VAL_AOS, nullptr, g.rows, 0} : Loader{LD_KEY32_VAL_SOA, nullptr, g.vals, 0};
    u32 *sorted_ids = nullptr;
    u64 *sorted_vals = nullptr;
    // 6. CSR offsets: recorded by the last sort pass itself when it runs as rp_gsweep_kernel<CSR> (offsets pre-set to all ones,
    //    offsets[D] = n), otherwise from the sorted ids
    DevBuf offs(c);
    TRY(offs.alloc((D + 1) * 8));
    CU(cudaMemsetAsync(offs.p, 0xFF, (D + 1) * 8, c->stream));
    bool csr_done = false;
    TRY(sort_id_pairs(s, ids.as<u32>(), first, n, ceil_log2_u64(std::max<u64>(D, 2)), &sorted_ids, &sorted_vals, dense.as<u32>(), offs.as<u64>(), &csr_done));
    DevBuf sid_guard(c);
    if (sorted_ids != ids.as<u32>()) sid_guard.p = sorted_ids;
    if (csr_done) {
        const u64 total = n;
        CU(cudaMemcpyAsync(offs.as<u64>() + D, &total, 8, cudaMemcpyHostToDevice, c->stream));   // pageable 8-byte source: copied before the call returns
    } else {
        KLaunch kl(s, K_MISC);
        u64 blocks = std::min<u64>((n + 255) / 256, (u64)c->sm_count * 8);
        csr_bounds_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(sorted_ids, n, offs.as<u64>(), D);
        TRY(kl.done("csr_bounds_kernel"));
    }
    // 7. value offsets at the partition boundaries
    {
        DevBuf idx(c), out(c);
        TRY(idx.alloc(((size_t)R + 1) * 8));
        TRY(out.alloc(((size_t)R + 1) * 8));
        CU(cudaMemcpyAsync(idx.p, s->bucket_off.data(), ((size_t)R + 1) * 8, cudaMemcpyHostToDevice, c->stream));
        KLaunch kl(s, K_MISC);
        gather_u64_kernel<<<(R + 1 + 255) / 256, 256, 0, c->stream>>>(offs.as<u64>(), idx.as<u64>(), R + 1, out.as<u64>());
        TRY(kl.done("gather_u64_kernel"));
        CU(cudaMemcpyAsync(s->val_off.data(), out.p, ((size_t)R + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
    }
    s->n_keys = D;
    s->n_vals = n;
    s->res_keys = (u64 *)ckeys.release();
    s->res_offs = (u64 *)offs.release();
    s->res_vals = sorted_vals;
    s->dense_of_slot = (u32 *)dense.release();
    s->st.rows_out = n;
    return VB_OK;
}

// Merge the per-map combined tables of this process into one (ShuffledRdd::compute's
// merge_combiners loop, shuffled_rdd.rs:154-164, for the partitions held locally).
// Settle the shared table of the borrowed-input map tasks: wait for the queued kernels, and if the table
// overflowed or a map id was resubmitted, rebuild it from the (still borrowed) inputs with build_table's
// restart logic.
static int settle_shared_table(vb_shuf *s, u64 *n_ins)
{
    vb_ctx *c = s->ctx;
    *n_ins = 0;
    bool any = false;
    for (auto &m : s->maps) any |= (m.present && m.in_shared && m.n_rows);
    bool rebuild = s->sh_dirty;
    if (s->sh_tab) {
        TableCtl *h = (TableCtl *)c->h_scratch;
        CU(cudaMemcpyAsync(h, s->sh_ctl, sizeof(TableCtl), cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        if (h->abort) { rebuild = true; s->st.table_restarts++; }
        *n_ins = h->n_inserted;
    }
    if (rebuild) {
        dev_free(c, s->sh_tab); dev_free(c, s->sh_ctl);
        s->sh_tab = nullptr; s->sh_ctl = nullptr;
        s->sh_dirty = false;
        if (any) {
            std::vector<AggInput> in;
            for (auto &m : s->maps)
                if (m.present && m.in_shared && m.n_rows)
                    in.push_back(AggInput{m.rows ? IN_AOS : IN_SOA, m.rows ? m.rows : m.keys, m.vals, m.n_rows, VB_DEVICE});
            TRY(build_table(s, K_HASH_AGG, in, map_opk(s), val_tx(s), std::max<u64>(s->hint, 2 * (*n_ins)), &s->sh_tab, &s->sh_log_cap, n_ins, nullptr));
        }
    }
    return VB_OK;
}

static int merge_map_tables(vb_shuf *s, void **tab, u32 *log_cap, u64 *n_ins)
{
    u64 sh_ins = 0;
    TRY(settle_shared_table(s, &sh_ins));
    struct T { void *tab; u32 log_cap; u64 ins; };
    std::vector<T> ts;
    if (s->sh_tab) ts.push_back(T{s->sh_tab, s->sh_log_cap, sh_ins});
    for (auto &m : s->maps) if (m.present && m.table) ts.push_back(T{m.table, m.log_cap, m.n_inserted});
    auto disown = [&]() {
        s->sh_tab = nullptr;
        dev_free(s->ctx, s->sh_ctl); s->sh_ctl = nullptr;
        for (auto &m : s->maps) m.table = nullptr;
    };
    if (ts.empty()) { *tab = nullptr; *log_cap = 0; *n_ins = 0; return VB_OK; }
    if (ts.size() == 1) {
        *tab = ts[0].tab; *log_cap = ts[0].log_cap; *n_ins = ts[0].ins;
        disown();
        return VB_OK;
    }
    std::vector<AggInput> in;
    u64 max_ins = 0;
    for (auto &t : ts) {
        const Table mt = table_at(t.tab, t.log_cap);
        in.push_back(AggInput{IN_TABLE, mt.keys, mt.accs, (1ull << t.log_cap) + 1, VB_DEVICE, t.ins + 1});
        max_ins = std::max(max_ins, t.ins);
    }
    TRY(build_table(s, K_MERGE, in, merge_opk(s), TX_NONE, std::max<u64>(max_ins, s->hint), tab, log_cap, n_ins, nullptr));
    for (auto &t : ts) dev_free(s->ctx, t.tab);
    disown();
    return VB_OK;
}

// Final (K, C) rows of a combined table, grouped by reduce partition.
static int finalize_reduce(vb_shuf *s, void *tab, u32 log_cap, u64 n_ins)
{
    vb_ctx *c = s->ctx;
    const u32 R = s->n_reduce;
    s->bucket_off.assign((size_t)R + 1, 0);
    s->val_off.assign((size_t)R + 1, 0);
    if (!tab) return VB_OK;
    const u64 cap = 1ull << log_cap;
    const u64 max_d = n_ins + 1;
    DevBuf k(c), v(c);
    TRY(k.alloc(max_d * 8));
    TRY(v.alloc(max_d * 8));
    const Table ft = table_at(tab, log_cap);
    Loader lt{LD_TABLE_KV, ft.keys, ft.accs, cap};
    static const bool ordered_only = getenv("VEGA_B200_STABLE_TABLE_SPLIT") != nullptr;     // A/B switch
    if (R <= (u32)TS_MAX_BINS && !ordered_only) TRY(multisplit_table_unordered(s, ft, DG_BUCKET, R, k.as<u64>(), v.as<u64>(), s->bucket_off));
    else TRY(multisplit(s, lt, cap + 1, DG_BUCKET, R, max_d, k.as<u64>(), v.as<u64>(), s->bucket_off));
    const u64 D = s->bucket_off[R];
    const int tx = val_tx(s);
    if (tx != TX_NONE && D) {
        KLaunch kl(s, K_MISC);
        tx_inv_kernel<<<(unsigned)((D + 255) / 256), 256, 0, c->stream>>>(v.as<u64>(), D, tx);
        TRY(kl.done("tx_inv_kernel"));
    }
    s->n_keys = D;
    s->res_keys = (u64 *)k.release();
    s->res_comb = (u64 *)v.release();
    s->st.rows_out = D;
    return VB_OK;
}

static int seal_sort(vb_shuf *s, const Gathered &g)
{
    vb_ctx *c = s->ctx;
    const u32 R = s->n_reduce;
    s->bucket_off.assign((size_t)R + 1, 0);
    s->val_off.assign((size_t)R + 1, 0);
    const u64 n = g.n;
    if (n == 0) return VB_OK;
    const bool has_val = g.rows != nullptr || g.vals != nullptr;
    const int tx = s->kdt == VB_I64 ? TX_I64 : s->kdt == VB_F64 ? TX_F64 : TX_NONE;
    DevBuf ka(c), kb(c), va(c), vbuf(c), hist(c);
    TRY(ka.alloc(n * 8));
    TRY(kb.alloc(n * 8));
    if (has_val) { TRY(va.alloc(n * 8)); TRY(vbuf.alloc(n * 8)); }
    u64 *src_k = nullptr, *src_v = nullptr, *dst_k = ka.as<u64>(), *dst_v = va.as<u64>();
    constexpr u32 SORT_PASSES = (64 + RP_SORT_BITS - 1) / RP_SORT_BITS;
    bool swept = false;
    {
        Loader l0 = g.rows ? Loader{LD_AOS64, g.rows, nullptr, 0} : Loader{LD_SOA64, g.keys, g.vals, 0};
        Digit dgp{};
        dgp.mode = DG_BITS; dgp.tx = tx;
        const bool ok = RP_SORT_BITS == 8 && (has_val ? sweep_applicable<u64, true>(l0, dgp, n) : sweep_applicable<u64, false>(l0, dgp, n));
        if (ok) {
            // sweep path: all 8 digit histograms from ONE read of the keys; a digit on which every key agrees (one bin
            // holds all n rows) needs no pass; then one look-back kernel per remaining digit
            DevBuf bases(c), scratch(c);
            TRY(bases.alloc((size_t)8 * SW_NB * 4));
            TRY(scratch.alloc(std::max(sweep_scratch_bytes<u64, true>(n), sweep_scratch_bytes<u64, false>(n))));
            HistAllArgs ha{};
            ha.n_pos = 8;
            for (u32 p = 0; p < 8; ++p) ha.shifts[p] = 8 * p;
            if (has_val) TRY((sweep_hist<u64, true>(s, l0, dgp, n, ha, bases.as<u32>())));
            else TRY((sweep_hist<u64, false>(s, l0, dgp, n, ha, bases.as<u32>())));
            u32 *hb = (u32 *)c->h_scratch;
            CU(cudaMemcpyAsync(hb, bases.p, 8 * SW_NB * 4, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            bool vary[8];
            u32 n_vary = 0;
            for (u32 p = 0; p < 8; ++p) {          // exclusive scan of a one-bin histogram: every base is 0 or n
                vary[p] = false;
                for (u32 d = 0; d < SW_NB; ++d) { const u32 b = hb[p * SW_NB + d]; if (b != 0 && b != (u32)n) { vary[p] = true; break; } }
                n_vary += vary[p];
            }
            if (n_vary == 0) vary[0] = true;      // at least one pass: it also copies the rows out
            bool first = true;
            for (u32 p = 0; p < 8; ++p) {
                if (!vary[p]) continue;
                Loader ld = first ? l0 : Loader{LD_SOA64, src_k, has_val ? src_v : nullptr, 0};
                first = false;
                Digit dg{};
                dg.mode = DG_BITS; dg.shift = 8 * p; dg.mask = 0xFF; dg.tx = tx;
                if (has_val) TRY((sweep_pass<u64, true>(s, ld, dg, n, dst_k, dst_v, bases.as<u32>() + (size_t)p * SW_NB, scratch.as<u32>())));
                else TRY((sweep_pass<u64, false>(s, ld, dg, n, dst_k, nullptr, bases.as<u32>() + (size_t)p * SW_NB, scratch.as<u32>())));
                u64 *nk = (src_k == nullptr) ? kb.as<u64>() : src_k;
                u64 *nv = (src_v == nullptr) ? vbuf.as<u64>() : src_v;
                src_k = dst_k; src_v = dst_v; dst_k = nk; dst_v = nv;
            }
            swept = true;
        }
    }
    PassPlan plan = has_val ? plan_pass<u64, true>(c, n, RP_SORT_BITS) : plan_pass<u64, false>(c, n, RP_SORT_BITS);
    if (!swept) TRY(hist.alloc(plan.hist_bytes()));
    // digits on which all keys agree are skipped (e.g. 32-bit-range keys take 4 passes, not 8)
    u64 varying = ~0ull;
    if (!swept) {
        DevBuf bits(c);
        TRY(bits.alloc(16));
        const unsigned long long init[2] = {0ull, ~0ull};
        CU(cudaMemcpyAsync(bits.p, init, 16, cudaMemcpyHostToDevice, c->stream));
        KLaunch kl(s, K_MISC);
        key_bits_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(g.rows ? g.rows : g.keys, g.rows ? 2 : 1, n, tx, (unsigned long long *)bits.p);
        TRY(kl.done("key_bits_kernel"));
        u64 *h = (u64 *)c->h_scratch;
        CU(cudaMemcpyAsync(h, bits.p, 16, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        varying = h[0] ^ h[1];
    }
    bool first = true;
    u32 done = 0;
    for (u32 p = 0; p < SORT_PASSES && !swept; ++p) {
        const u64 dmask = (u64)((1u << RP_SORT_BITS) - 1) << (RP_SORT_BITS * p);
        const bool last_chance = (p + 1 == SORT_PASSES) && done == 0;      // at least one pass: it also copies the rows out
        if (!(varying & dmask) && !last_chance) continue;
        ++done;
        Loader ld;
        if (first) ld = g.rows ? Loader{LD_AOS64, g.rows, nullptr, 0} : Loader{LD_SOA64, g.keys, g.vals, 0};
        else ld = Loader{LD_SOA64, src_k, has_val ? src_v : nullptr, 0};
        first = false;
        Digit dg{};
        dg.mode = DG_BITS; dg.shift = RP_SORT_BITS * p; dg.mask = (1u << RP_SORT_BITS) - 1; dg.tx = tx;
        if (has_val) TRY((radix_pass<u64, true>(s, ld, dg, n, dst_k, dst_v, hist.as<u32>(), plan)));
        else TRY((radix_pass<u64, false>(s, ld, dg, n, dst_k, nullptr, hist.as<u32>(), plan)));
        u64 *nk = (src_k == nullptr) ? kb.as<u64>() : src_k;
        u64 *nv = (src_v == nullptr) ? vbuf.as<u64>() : src_v;
        src_k = dst_k; src_v = dst_v; dst_k = nk; dst_v = nv;
    }
    // results are in the buffer written by the last pass (ka, kb alternate starting with ka)
    DevBuf starts(c);
    TRY(starts.alloc(((size_t)R + 1) * 8));
    {
        KLaunch kl(s, K_MISC);
        sort_cuts_kernel<<<(R + 1 + 255) / 256, 256, 0, c->stream>>>(src_k, n, R, starts.as<u64>());
        TRY(kl.done("sort_cuts_kernel"));
    }
    CU(cudaMemcpyAsync(s->bucket_off.data(), starts.p, ((size_t)R + 1) * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    s->n_keys = n;
    s->res_keys = src_k;
    s->res_comb = has_val ? src_v : nullptr;
    if (src_k == ka.as<u64>()) ka.release(); else kb.release();
    if (has_val) { if (src_v == va.as<u64>()) va.release(); else vbuf.release(); }
    s->st.rows_out = n;
    return VB_OK;
}

static void release_inputs(vb_shuf *s)
{
    dev_free(s->ctx, s->sh_tab); dev_free(s->ctx, s->sh_ctl);
    s->sh_tab = nullptr; s->sh_ctl = nullptr;
    for (auto &m : s->maps) if (m.present) { u64 n = m.n_rows; free_map(s, m); m.present = true; m.n_rows = n; }
    dev_free(s->ctx, s->gath_keys);
    dev_free(s->ctx, s->gath_vals);
    s->gath_keys = s->gath_vals = nullptr;
    dev_free(s->ctx, s->exp_keys);
    dev_free(s->ctx, s->exp_vals);
    dev_free(s->ctx, s->exp_hist);
    s->exp_keys = s->exp_vals = nullptr;
    s->exp_hist = nullptr;
    dev_free(s->ctx, s->imp_own_k);
    dev_free(s->ctx, s->imp_own_v);
    s->imp_own_k = s->imp_own_v = nullptr;
}

// Finish the local map side and pack rows by destination rank (caller holds c->mu).
static int export_prepare_locked(vb_shuf *s, uint64_t *counts)
{
    vb_ctx *c = s->ctx;
    {
        std::lock_guard<std::mutex> g(s->mu);
        if (s->sealed || s->exported || s->freed) return set_err(VB_ERR_STATE, "export after seal/export");
    }
    std::vector<u64> off;
    if (is_reduce_op(s->agg)) {
        void *tab = nullptr; u32 log_cap = 0; u64 n_ins = 0;
        TRY(merge_map_tables(s, &tab, &log_cap, &n_ins));
        off.assign((size_t)s->world + 1, 0);
        if (tab) {
            DevBuf guard(c); guard.p = tab;
            DevBuf k(c), v(c);
            TRY(k.alloc((n_ins + 1) * 8));
            TRY(v.alloc((n_ins + 1) * 8));
            const Table et = table_at(tab, log_cap);
            Loader lt{LD_TABLE_KV, et.keys, et.accs, 1ull << log_cap};
            static const bool ordered_only = getenv("VEGA_B200_STABLE_TABLE_SPLIT") != nullptr;
            if (s->world <= (u32)TS_MAX_BINS && !ordered_only) TRY(multisplit_table_unordered(s, et, DG_DEST, s->world, k.as<u64>(), v.as<u64>(), off));
            else TRY(multisplit(s, lt, (1ull << log_cap) + 1, DG_DEST, s->world, n_ins + 1, k.as<u64>(), v.as<u64>(), off));
            s->exp_keys = (u64 *)k.release();
            s->exp_vals = (u64 *)v.release();
        }
    } else {
        Gathered g;
        TRY(gather_maps(s, &g));
        off.assign((size_t)s->world + 1, 0);
        if (g.n) {
            DevBuf k(c), v(c);
            TRY(k.alloc(g.n * 8));
            TRY(v.alloc(g.n * 8));
            Loader ld = g.rows ? Loader{LD_AOS64, g.rows, nullptr, 0} : Loader{LD_SOA64, g.keys, g.vals, 0};
            TRY(multisplit(s, ld, g.n, DG_DEST, s->world, g.n, k.as<u64>(), v.as<u64>(), off));
            s->exp_keys = (u64 *)k.release();
            s->exp_vals = (u64 *)v.release();
        }
    }
    for (u32 r = 0; r < s->world; ++r) counts[r] = off[r + 1] - off[r];
    std::lock_guard<std::mutex> g(s->mu);
    s->exported = true;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_export_prepare(vb_shuf *s, uint64_t *counts)
{
    if (!s || !counts) return set_err(VB_ERR_INVALID, "NULL argument");
    if (s->world < 2) return set_err(VB_ERR_STATE, "vb_shuffle_export_prepare needs vb_shuffle_set_dist(world > 1)");
    vb_ctx *c = s->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    TRY(export_prepare_locked(s, counts));
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// P2P exchange: rows go straight from the partition kernel into the peers' HBM over NVLink
// ---------------------------------------------------------------------------------------------
static int arena_reserve_locked(vb_ctx *c, uint64_t bytes, void *handle_out, uint64_t *generation)
{
    if (bytes > c->arena_bytes || !c->arena) {
        CU(cudaStreamSynchronize(c->stream));
        // peers may still have the old allocation mapped (they close it in vb_ctx_peer_open when they see the new
        // generation): keep it until vb_ctx_arena_release_retired, which the caller invokes after a barrier
        if (c->arena) c->retired_arenas.push_back(c->arena);
        c->arena = nullptr;
        size_t want = std::max<size_t>((size_t)bytes + bytes / 4, (size_t)64 << 20);
        want = (want + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
        CU(cudaMalloc(&c->arena, want));     // cudaMalloc, not the async pool: legacy IPC handles need it
        c->arena_bytes = want;
        c->arena_gen++;
    }
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, c->arena));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle_out, &h, sizeof(h));
    *generation = c->arena_gen;
    return VB_OK;
}

extern "C" int32_t vb_ctx_arena_reserve(vb_ctx *c, uint64_t bytes, void *handle_out, uint64_t *generation)
{
    if (!c || !handle_out || !generation) return set_err(VB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    return arena_reserve_locked(c, bytes, handle_out, generation);
}

// Free the arenas outgrown by vb_ctx_arena_reserve.  Contract: every peer has called vb_ctx_peer_open with this
// rank's current generation (which closes its mapping of the old one) — i.e. call it after the barrier that
// follows the exchange.
extern "C" int32_t vb_ctx_arena_release_retired(vb_ctx *c)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    for (void *p : c->retired_arenas) CU(cudaFree(p));
    c->retired_arenas.clear();
    return VB_OK;
}

static int peer_open_locked(vb_ctx *c, uint32_t peer_rank, const void *handle, uint64_t generation, int32_t is_self)
{
    auto &p = c->peers[peer_rank];
    if (is_self) { p.base = c->arena; p.gen = c->arena_gen; p.self = true; return VB_OK; }
    if (p.base && p.gen == generation && !p.self) return VB_OK;
    if (p.base && !p.self) { CU(cudaStreamSynchronize(c->stream)); cudaIpcCloseMemHandle(p.base); p.base = nullptr; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    void *base = nullptr;
    CU(cudaIpcOpenMemHandle(&base, h, cudaIpcMemLazyEnablePeerAccess));
    p.base = base; p.gen = generation; p.self = false;
    return VB_OK;
}

extern "C" int32_t vb_ctx_peer_open(vb_ctx *c, uint32_t peer_rank, const void *handle, uint64_t generation, int32_t is_self)
{
    if (!c || (!handle && !is_self)) return set_err(VB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    return peer_open_locked(c, peer_rank, handle, generation, is_self);
}

// Histogram of this rank's rows by destination rank (no data movement yet); keeps the scanned
// per-part histogram for vb_shuffle_export_direct.  group ops only (reduce ops exchange a few MB of
// combined rows: vb_shuffle_export_prepare + one all-to-all-v is the right tool there).
static int export_counts_locked(vb_shuf *s, uint64_t *counts)
{
    if (!is_group_op(s->agg)) return set_err(VB_ERR_UNSUPPORTED, "the fused P2P export is for GROUP/COGROUP shuffles");
    vb_ctx *c = s->ctx;
    {
        std::lock_guard<std::mutex> g(s->mu);
        if (s->sealed || s->exported || s->exp_counted || s->freed) return set_err(VB_ERR_STATE, "export after seal/export");
    }
    Gathered g;
    TRY(gather_maps(s, &g));
    s->exp_rows = g.rows; s->exp_k = g.keys; s->exp_v = g.vals; s->exp_n = g.n;
    s->exp_digit_start.assign((size_t)s->world + 1, 0);
    if (g.n) {
        PassPlan plan = plan_pass<u64, true>(c, g.n, 8);
        DevBuf hist(c);
        TRY(hist.alloc(plan.hist_bytes()));
        Loader ld = g.rows ? Loader{LD_AOS64, g.rows, nullptr, 0} : Loader{LD_SOA64, g.keys, g.vals, 0};
        Digit dg = make_bucket_digit(s, DG_DEST, 0, 0xFFFFFFFFu);
        TRY((radix_hist_scan<u64>(s, ld, dg, g.n, hist.as<u32>(), plan)));
        TRY(fetch_offsets(c, hist.as<u32>(), plan, s->world, s->exp_digit_start.data()));
        s->exp_hist = (u32 *)hist.release();
        s->exp_parts = plan.num_parts;
        s->exp_rows_per_part = plan.rows_per_part;
    }
    for (u32 r = 0; r < s->world; ++r) counts[r] = s->exp_digit_start[r + 1] - s->exp_digit_start[r];
    std::lock_guard<std::mutex> gg(s->mu);
    s->exp_counted = true;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_export_counts(vb_shuf *s, uint64_t *counts)
{
    if (!s || !counts) return set_err(VB_ERR_INVALID, "NULL argument");
    if (s->world < 2) return set_err(VB_ERR_STATE, "vb_shuffle_export_counts needs vb_shuffle_set_dist(world > 1)");
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    CU(cudaSetDevice(s->ctx->device));
    return export_counts_locked(s, counts);
}

// The scatter: every row is stored into the arena of the rank that owns its reduce partition.
// dst_row_offset[d]: first row of my block inside rank d's arena; dst_total_rows[d]: rows rank d receives in total
// (its arena holds keys[total] then vals[total]).  Returns after the stores are complete on this GPU; the
// host then barriers the ranks before anyone reads its arena.
static int export_direct_locked(vb_shuf *s, const uint64_t *dst_row_offset, const uint64_t *dst_total_rows, bool sync)
{
    if (!s->exp_counted || s->exported) return set_err(VB_ERR_STATE, "vb_shuffle_export_direct needs vb_shuffle_export_counts first");
    vb_ctx *c = s->ctx;
    const u32 W = s->world;
    if (s->exp_n) {
        std::vector<u64 *> hk(W), hv(W);
        std::vector<u32> hadj(W);
        for (u32 d = 0; d < W; ++d) {
            auto it = c->peers.find(d);
            const u64 cnt = s->exp_digit_start[d + 1] - s->exp_digit_start[d];
            if (it == c->peers.end() || !it->second.base) {
                if (cnt) return set_err(VB_ERR_STATE, "peer %u arena not opened (vb_ctx_peer_open)", d);
                hk[d] = hv[d] = nullptr; hadj[d] = 0;
                continue;
            }
            if (dst_row_offset[d] + cnt > dst_total_rows[d] || dst_total_rows[d] >= 0xFFFFFFFFull)
                return set_err(VB_ERR_INVALID, "bad arena layout for destination %u", d);
            hk[d] = (u64 *)it->second.base;
            hv[d] = hk[d] + dst_total_rows[d];
            hadj[d] = (u32)(dst_row_offset[d] - s->exp_digit_start[d]);
        }
        DevBuf dk(c), dv(c), da(c);
        TRY(dk.alloc(W * 8)); TRY(dv.alloc(W * 8)); TRY(da.alloc(W * 4));
        CU(cudaMemcpyAsync(dk.p, hk.data(), W * 8, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(dv.p, hv.data(), W * 8, cudaMemcpyHostToDevice, c->stream));
        CU(cudaMemcpyAsync(da.p, hadj.data(), W * 4, cudaMemcpyHostToDevice, c->stream));
        Loader ld = s->exp_rows ? Loader{LD_AOS64, s->exp_rows, nullptr, 0} : Loader{LD_SOA64, s->exp_k, s->exp_v, 0};
        Digit dg = make_bucket_digit(s, DG_DEST, 0, 0xFFFFFFFFu);
        const void *sk = s->exp_rows ? (const void *)rp_scatter_kernel<u64, true, LD_AOS64, DG_DEST, 8, true>
                                     : (const void *)rp_scatter_kernel<u64, true, LD_SOA64, DG_DEST, 8, true>;
        const size_t smem = scatter_smem<u64, true>(8);
        CU(cudaFuncSetAttribute(sk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        u64 n = s->exp_n, rpp = s->exp_rows_per_part;
        u32 np = s->exp_parts;
        const u32 *ch = s->exp_hist;
        u64 *nullk = nullptr, *nullv = nullptr;
        RemoteDst rd{dk.as<u64 *>(), dv.as<u64 *>(), da.as<u32>(), W};
        KLaunch kl(s, K_RP_SCATTER, n);
        void *args[] = {&ld, &dg, &n, &rpp, &ch, &np, &nullk, &nullv, &rd};
        CU(cudaLaunchKernel(sk, dim3(np), dim3(RPS_THREADS), args, smem, c->stream));
        TRY(kl.done("rp_scatter_kernel<REMOTE>"));
        if (sync) CU(cudaStreamSynchronize(c->stream));
    }
    dev_free(c, s->exp_hist);
    s->exp_hist = nullptr;
    std::lock_guard<std::mutex> g(s->mu);
    s->exported = true;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_export_direct(vb_shuf *s, const uint64_t *dst_row_offset, const uint64_t *dst_total_rows)
{
    if (!s || !dst_row_offset || !dst_total_rows) return set_err(VB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    CU(cudaSetDevice(s->ctx->device));
    return export_direct_locked(s, dst_row_offset, dst_total_rows, true);
}

// The rows of every source rank are already in this context's arena (keys[total] then vals[total],
// source-rank major): hand them to the reduce side.  counts[world] as in vb_shuffle_import.
extern "C" int32_t vb_shuffle_import_arena(vb_shuf *s, const uint64_t *counts)
{
    if (!s || !counts) return set_err(VB_ERR_INVALID, "NULL argument");
    if (!s->exported || s->sealed) return set_err(VB_ERR_STATE, "import needs the export first and no seal yet");
    u64 n = 0;
    for (u32 r = 0; r < s->world; ++r) n += counts[r];
    if (n * 16 > s->ctx->arena_bytes) return set_err(VB_ERR_INVALID, "arena holds %zu bytes, %llu rows announced", s->ctx->arena_bytes, (unsigned long long)n);
    if (n >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "import of %llu rows", (unsigned long long)n);
    s->imp_keys = (const u64 *)s->ctx->arena;
    s->imp_vals = s->imp_keys + n;
    s->imp_n = n;
    s->imported = true;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_export_buffers(vb_shuf *s, void **keys_dev, void **vals_dev)
{
    if (!s || !keys_dev || !vals_dev) return set_err(VB_ERR_INVALID, "NULL argument");
    if (!s->exported) return set_err(VB_ERR_STATE, "vb_shuffle_export_buffers before vb_shuffle_export_prepare");
    *keys_dev = s->exp_keys;
    *vals_dev = s->exp_vals;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_import(vb_shuf *s, const void *keys_dev, const void *vals_dev, const uint64_t *counts)
{
    if (!s || !counts) return set_err(VB_ERR_INVALID, "NULL argument");
    if (!s->exported || s->sealed) return set_err(VB_ERR_STATE, "import needs export_prepare first and no seal yet");
    u64 n = 0;
    for (u32 r = 0; r < s->world; ++r) n += counts[r];
    if (n && (!keys_dev || !vals_dev)) return set_err(VB_ERR_INVALID, "NULL buffers with rows to import");
    if (n >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "import of %llu rows", (unsigned long long)n);
    s->imp_keys = (const u64 *)keys_dev;
    s->imp_vals = (const u64 *)vals_dev;
    s->imp_n = n;
    s->imported = true;
    return VB_OK;
}


// ---------------------------------------------------------------------------------------------
// The exchange behind the C ABI (ShuffleFetcher::fetch, src/shuffle/shuffle_fetcher.rs:16-119):
// one NCCL communicator per context, counts + rows exchanged on the library's own stream.
// NCCL is loaded with dlopen on first use, so single-GPU users carry no dependency on it.
// ---------------------------------------------------------------------------------------------
#include <dlfcn.h>
#include <nccl.h>

struct NcclApi {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;
};
static NcclApi g_nccl;
static std::mutex g_nccl_mu;

static int nccl_load()
{
    std::lock_guard<std::mutex> g(g_nccl_mu);
    if (g_nccl.h) return VB_OK;
    const char *names[] = {getenv("VEGA_B200_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *nm : names) {
        if (!nm) continue;
        h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) return set_err(VB_ERR_UNSUPPORTED, "NCCL not found (dlopen libnccl.so.2): %s", dlerror());
#define LD(f)                                                                                      \
    do {                                                                                           \
        *(void **)(&g_nccl.f) = dlsym(h, "nccl" #f);                                               \
        if (!g_nccl.f) return set_err(VB_ERR_UNSUPPORTED, "libnccl lacks nccl" #f);                \
    } while (0)
    LD(GetUniqueId); LD(CommInitRank); LD(CommDestroy); LD(GroupStart); LD(GroupEnd); LD(Send); LD(Recv); LD(AllGather);
    LD(GetErrorString); LD(GetVersion);
#undef LD
    g_nccl.h = h;
    return VB_OK;
}

#define NC(expr)                                                                                             \
    do {                                                                                                     \
        ncclResult_t r_ = (expr);                                                                            \
        if (r_ != ncclSuccess) return set_err(VB_ERR_CUDA, "%s:%d %s: NCCL %s", __FILE__, __LINE__, #expr,    \
                                              g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "error");   \
    } while (0)

struct Comm {
    ncclComm_t comm = nullptr;
    u32 rank = 0, world = 1;
    u64 *d_send = nullptr;     // [world + 2]: counts to every destination, arena bytes, arena generation
    u64 *d_recv = nullptr;     // [world][world + 2]
    unsigned char *d_hs = nullptr, *d_hr = nullptr;   // IPC handle + generation: 80 bytes, [world] x 80
    std::vector<u64> peer_arena_bytes, peer_gen_seen;
    bool handles_valid = false;
};
constexpr u32 COMM_MAX_WORLD = 64;
constexpr size_t COMM_HOST_OFF = 256 << 10;   // staging region inside vb_ctx::h_scratch

static void comm_teardown(vb_ctx *c)
{
    Comm *m = c->comm;
    if (!m) return;
    // every rank has closed its peer mappings before this point; the all-gather is the barrier that lets the
    // owners free the exported arenas afterwards
    if (m->comm && g_nccl.AllGather && m->d_send && m->d_recv) {
        if (g_nccl.AllGather(m->d_send, m->d_recv, 1, ncclUint64, m->comm, c->stream) == ncclSuccess) cudaStreamSynchronize(c->stream);
    }
    if (m->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(m->comm);
    cudaFree(m->d_send); cudaFree(m->d_recv); cudaFree(m->d_hs); cudaFree(m->d_hr);
    cudaGetLastError();
    delete m;
    c->comm = nullptr;
}

extern "C" int32_t vb_comm_unique_id(void *id_out)
{
    if (!id_out) return set_err(VB_ERR_INVALID, "id_out is NULL");
    TRY(nccl_load());
    static_assert(sizeof(ncclUniqueId) == VB_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NC(g_nccl.GetUniqueId(&id));
    memcpy(id_out, &id, sizeof(id));
    return VB_OK;
}

extern "C" int32_t vb_ctx_comm_init(vb_ctx *c, const void *unique_id, uint32_t rank, uint32_t world)
{
    if (!c || !unique_id) return set_err(VB_ERR_INVALID, "NULL argument");
    if (world < 1 || rank >= world || world > COMM_MAX_WORLD) return set_err(VB_ERR_INVALID, "bad rank/world (world <= %u)", COMM_MAX_WORLD);
    TRY(nccl_load());
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    if (c->comm) return set_err(VB_ERR_STATE, "context already has a communicator");
    Comm *m = new Comm();
    m->rank = rank; m->world = world;
    ncclUniqueId id;
    memcpy(&id, unique_id, sizeof(id));
    ncclResult_t r = g_nccl.CommInitRank(&m->comm, (int)world, id, (int)rank);
    if (r != ncclSuccess) { delete m; return set_err(VB_ERR_CUDA, "ncclCommInitRank: %s", g_nccl.GetErrorString(r)); }
    c->comm = m;
    CU(cudaMalloc((void **)&m->d_send, (world + 2) * 8));
    CU(cudaMalloc((void **)&m->d_recv, (size_t)world * (world + 2) * 8));
    CU(cudaMalloc((void **)&m->d_hs, 80));
    CU(cudaMalloc((void **)&m->d_hr, (size_t)world * 80));
    CU(cudaMemset(m->d_send, 0, (world + 2) * 8));
    m->peer_arena_bytes.assign(world, 0);
    m->peer_gen_seen.assign(world, 0);
    return VB_OK;
}

extern "C" int32_t vb_ctx_comm_destroy(vb_ctx *c)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    CU(cudaStreamSynchronize(c->stream));
    for (auto &kv : c->peers) if (kv.second.base && !kv.second.self) { cudaIpcCloseMemHandle(kv.second.base); kv.second.base = nullptr; }
    c->peers.clear();
    comm_teardown(c);
    return VB_OK;
}

extern "C" int32_t vb_ctx_comm_info(vb_ctx *c, uint32_t *rank, uint32_t *world, int32_t *nccl_version)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    if (!c->comm) return set_err(VB_ERR_STATE, "no communicator (vb_ctx_comm_init)");
    if (rank) *rank = c->comm->rank;
    if (world) *world = c->comm->world;
    if (nccl_version) { int v = 0; g_nccl.GetVersion(&v); *nccl_version = v; }
    return VB_OK;
}

// All-gather of (counts[world], my arena bytes, my arena generation) — ONE small collective + one D2H —
// into the pinned staging area.  Returns the matrix as host rows of (world + 2) u64.
static int comm_gather_counts(vb_ctx *c, const u64 *counts, const u64 **matrix)
{
    Comm *m = c->comm;
    const u32 W = m->world;
    u64 *h = (u64 *)((char *)c->h_scratch + COMM_HOST_OFF);
    u64 *hs = h + (size_t)W * (W + 2);
    for (u32 d = 0; d < W; ++d) hs[d] = counts[d];
    hs[W] = c->arena_bytes;
    hs[W + 1] = c->arena_gen;
    CU(cudaMemcpyAsync(m->d_send, hs, (W + 2) * 8, cudaMemcpyHostToDevice, c->stream));
    NC(g_nccl.AllGather(m->d_send, m->d_recv, W + 2, ncclUint64, m->comm, c->stream));
    CU(cudaMemcpyAsync(h, m->d_recv, (size_t)W * (W + 2) * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *matrix = h;
    return VB_OK;
}

// reduce ops and non-P2P group ops: pack by destination, then ONE grouped send/recv carrying both columns
static int exchange_nccl_locked(vb_shuf *s)
{
    vb_ctx *c = s->ctx;
    Comm *m = c->comm;
    const u32 W = m->world, me = m->rank;
    std::vector<u64> counts(W, 0);
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto ms_since = [](std::chrono::steady_clock::time_point t0) { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    auto t0 = now();
    TRY(export_prepare_locked(s, counts.data()));
    s->xst.prepare_wall_ms += ms_since(t0);
    t0 = now();
    const u64 *mat = nullptr;
    TRY(comm_gather_counts(c, counts.data(), &mat));
    s->xst.counts_wall_ms += ms_since(t0);
    t0 = now();
    std::vector<u64> rcnt(W), soff(W + 1, 0), roff(W + 1, 0);
    for (u32 p = 0; p < W; ++p) {
        rcnt[p] = mat[(size_t)p * (W + 2) + me];
        soff[p + 1] = soff[p] + counts[p];
        roff[p + 1] = roff[p] + rcnt[p];
    }
    const u64 n_recv = roff[W];
    if (n_recv >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "rank %u would receive %llu rows", me, (unsigned long long)n_recv);
    DevBuf rk(c), rv(c);
    TRY(rk.alloc(std::max<u64>(n_recv, 1) * 8));
    TRY(rv.alloc(std::max<u64>(n_recv, 1) * 8));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (c->profile) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, c->stream); }
    NC(g_nccl.GroupStart());
    for (u32 p = 0; p < W; ++p) {
        if (counts[p]) {
            NC(g_nccl.Send(s->exp_keys + soff[p], counts[p], ncclUint64, (int)p, m->comm, c->stream));
            NC(g_nccl.Send(s->exp_vals + soff[p], counts[p], ncclUint64, (int)p, m->comm, c->stream));
        }
        if (rcnt[p]) {
            NC(g_nccl.Recv(rk.as<u64>() + roff[p], rcnt[p], ncclUint64, (int)p, m->comm, c->stream));
            NC(g_nccl.Recv(rv.as<u64>() + roff[p], rcnt[p], ncclUint64, (int)p, m->comm, c->stream));
        }
    }
    NC(g_nccl.GroupEnd());
    if (e0) {       // resolved later (vb_shuffle_exchange_stats / vb_shuffle_stats): no host wait here
        cudaEventRecord(e1, c->stream);
        s->timers.push_back(Timer{e0, e1, -3, 0});
    }
    s->xst.post_wall_ms += ms_since(t0);
    s->xst.sent_rows += soff[W] - counts[me];
    s->xst.recv_rows += n_recv - rcnt[me];
    s->xst.exchanges += 1;
    s->xst.kind = VB_XCHG_NCCL;
    s->imp_own_k = (u64 *)rk.release();
    s->imp_own_v = (u64 *)rv.release();
    s->imp_keys = s->imp_own_k; s->imp_vals = s->imp_own_v; s->imp_n = n_recv;
    s->imported = true;
    return VB_OK;
}

// group ops: the destination-rank partition kernel stores straight into the owners' arenas (peer memory)
static int exchange_p2p_locked(vb_shuf *s)
{
    vb_ctx *c = s->ctx;
    Comm *m = c->comm;
    const u32 W = m->world, me = m->rank;
    std::vector<u64> counts(W, 0);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (c->profile) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, c->stream); }
    TRY(export_counts_locked(s, counts.data()));
    const u64 *mat = nullptr;
    TRY(comm_gather_counts(c, counts.data(), &mat));
    // arena layout (source-rank major = map-id order) from the count matrix
    std::vector<u64> total(W, 0), my_off(W, 0), rcnt(W);
    for (u32 dst = 0; dst < W; ++dst)
        for (u32 src = 0; src < W; ++src) {
            const u64 x = mat[(size_t)src * (W + 2) + dst];
            if (src < me) my_off[dst] += x;
            total[dst] += x;
        }
    for (u32 src = 0; src < W; ++src) rcnt[src] = mat[(size_t)src * (W + 2) + me];
    // who must (re)grow its arena is a pure function of the gathered matrix: handles are re-exchanged only then
    bool any_regrow = !m->handles_valid;
    for (u32 p = 0; p < W; ++p) {
        const u64 need = 16 * std::max<u64>(total[p], 1), have = mat[(size_t)p * (W + 2) + W], gen = mat[(size_t)p * (W + 2) + W + 1];
        if (need > have || gen == 0 || gen != m->peer_gen_seen[p]) any_regrow = true;
    }
    unsigned char hbuf[80];
    u64 gen = 0;
    TRY(arena_reserve_locked(c, 16 * std::max<u64>(total[me], 1), hbuf, &gen));
    if (any_regrow) {
        memcpy(hbuf + 64, &gen, 8);
        memset(hbuf + 72, 0, 8);
        unsigned char *hh = (unsigned char *)c->h_scratch + COMM_HOST_OFF + 128 * 1024;
        memcpy(hh, hbuf, 80);
        CU(cudaMemcpyAsync(m->d_hs, hh, 80, cudaMemcpyHostToDevice, c->stream));
        NC(g_nccl.AllGather(m->d_hs, m->d_hr, 80, ncclUint8, m->comm, c->stream));
        CU(cudaMemcpyAsync(hh + 128, m->d_hr, (size_t)W * 80, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        for (u32 p = 0; p < W; ++p) {
            u64 pg;
            memcpy(&pg, hh + 128 + (size_t)p * 80 + 64, 8);
            TRY(peer_open_locked(c, p, hh + 128 + (size_t)p * 80, pg, p == me));
            m->peer_gen_seen[p] = pg;
        }
        m->handles_valid = true;
    }
    TRY(export_direct_locked(s, my_off.data(), total.data(), false));
    // stream-ordered barrier: every rank's stores precede its part of this collective, which precedes my reads
    NC(g_nccl.AllGather(m->d_send, m->d_recv, 1, ncclUint64, m->comm, c->stream));
    if (any_regrow) {       // every peer has re-opened: outgrown arenas can go
        CU(cudaStreamSynchronize(c->stream));
        for (void *p : c->retired_arenas) CU(cudaFree(p));
        c->retired_arenas.clear();
    }
    u64 n = 0;
    for (u32 r = 0; r < W; ++r) n += rcnt[r];
    if (n >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "import of %llu rows", (unsigned long long)n);
    s->imp_keys = (const u64 *)c->arena;
    s->imp_vals = s->imp_keys + n;
    s->imp_n = n;
    s->imported = true;
    if (e0) {
        cudaEventRecord(e1, c->stream);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        s->xst.exchange_ms += ms;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    u64 sent = 0;
    for (u32 p = 0; p < W; ++p) if (p != me) sent += counts[p];
    s->xst.sent_rows += sent;
    s->xst.recv_rows += n - rcnt[me];
    s->xst.exchanges += 1;
    s->xst.kind = VB_XCHG_P2P;
    return VB_OK;
}


// ---- multi-rank sort_by_key -----------------------------------------------------------------------------------
// (no reference code: sort_by_key is absent from vega, SURVEY.md F2 — semantics = the single-GPU ones: output
// partition p is the p-th contiguous key range, cut at floor(p*N/R) moved past equal keys, stable.)
// Every rank sorts its rows locally, the ranks find the EXACT global cut keys by bisection over the key space
// (64 rounds, each one tiny all-gather of R-1 counts obtained by binary search in the sorted local run), each
// rank's sorted run is then cut into contiguous segments that travel in ONE grouped send/recv to the owners
// (partition p lives on rank p % world), and the owner's seal re-sorts what it received (stable: source-rank-major
// arrival order = map-id order).
__global__ void count_le_kernel(const u64 *__restrict__ sorted, u64 n, int tx, const u64 *__restrict__ cand, u32 m, u64 *__restrict__ out)
{
    const u32 p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= m) return;
    const u64 v = cand[p];
    u64 lo = 0, hi = n;                       // first index whose transformed key is > v
    while (lo < hi) {
        const u64 mid = lo + ((hi - lo) >> 1);
        if (tx_fwd(sorted[mid], tx) <= v) lo = mid + 1; else hi = mid;
    }
    out[p] = lo;
}

static int exchange_sort_locked(vb_shuf *s)
{
    vb_ctx *c = s->ctx;
    Comm *m = c->comm;
    const u32 W = m->world, me = m->rank, R = s->n_reduce;
    if (R > 4096) return set_err(VB_ERR_UNSUPPORTED, "multi-rank sort_by_key supports up to 4096 output partitions");
    {
        std::lock_guard<std::mutex> g(s->mu);
        if (s->sealed || s->exported || s->freed) return set_err(VB_ERR_STATE, "export after seal/export");
    }
    const int tx = s->kdt == VB_I64 ? TX_I64 : s->kdt == VB_F64 ? TX_F64 : TX_NONE;
    // 1. local sort
    Gathered g;
    TRY(gather_maps(s, &g));
    const bool has_val = g.rows != nullptr || g.vals != nullptr;
    TRY(seal_sort(s, g));
    const u64 n_local = g.n;
    u64 *lk = s->res_keys, *lv = s->res_comb;
    s->res_keys = s->res_comb = nullptr; s->n_keys = 0;
    DevBuf lk_guard(c), lv_guard(c);
    lk_guard.p = lk; lv_guard.p = lv;
    // every rank must agree on whether a payload travels (a rank with zero rows has no way to know locally)
    std::vector<u64> c0(W, 0);
    c0[0] = n_local; if (W > 1) c0[1] = has_val ? 1 : 0;
    const u64 *mat = nullptr;
    TRY(comm_gather_counts(c, c0.data(), &mat));
    u64 N = 0; bool any_val = false;
    for (u32 r = 0; r < W; ++r) { N += mat[(size_t)r * (W + 2)]; if (W > 1 && mat[(size_t)r * (W + 2)] && mat[(size_t)r * (W + 2) + 1]) any_val = true; }
    // 2. exact cut keys: s_p = the key of global rank c_p - 1, c_p = floor(p N / R); rows with key <= s_p go to partitions < p
    const u32 P = R - 1;
    std::vector<u64> need(P), lo(P, 0), hi(P, ~0ull), cut(R + 1, 0);
    std::vector<char> none(P, 0);
    for (u32 p = 1; p < R; ++p) {
        const u64 cp = (u64)(((unsigned __int128)p * N) / R);
        need[p - 1] = cp;                     // need count_le(v) >= c_p  (i.e. >= (c_p - 1) + 1)
        none[p - 1] = (cp == 0);
    }
    DevBuf d_cand(c), d_cnt(c), d_all(c);
    std::vector<u64> h_all((size_t)W * std::max<u32>(P, 1));
    if (P) {
        TRY(d_cand.alloc((size_t)P * 8)); TRY(d_cnt.alloc((size_t)P * 8)); TRY(d_all.alloc((size_t)W * P * 8));
        std::vector<u64> mid(P);
        for (int round = 0; round <= 64; ++round) {
            const bool final_round = (round == 64);
            for (u32 i = 0; i < P; ++i) mid[i] = final_round ? lo[i] : lo[i] + ((hi[i] - lo[i]) >> 1);
            CU(cudaMemcpyAsync(d_cand.p, mid.data(), (size_t)P * 8, cudaMemcpyHostToDevice, c->stream));
            {
                KLaunch kl(s, K_MISC);
                count_le_kernel<<<(P + 127) / 128, 128, 0, c->stream>>>(lk, n_local, tx, d_cand.as<u64>(), P, d_cnt.as<u64>());
                TRY(kl.done("count_le_kernel"));
            }
            if (final_round) {                 // local cut positions for the agreed cut keys
                CU(cudaMemcpyAsync(h_all.data(), d_cnt.p, (size_t)P * 8, cudaMemcpyDeviceToHost, c->stream));
                CU(cudaStreamSynchronize(c->stream));
                for (u32 i = 0; i < P; ++i) cut[i + 1] = none[i] ? 0 : h_all[i];
                break;
            }
            NC(g_nccl.AllGather(d_cnt.p, d_all.p, P, ncclUint64, m->comm, c->stream));
            CU(cudaMemcpyAsync(h_all.data(), d_all.p, (size_t)W * P * 8, cudaMemcpyDeviceToHost, c->stream));
            CU(cudaStreamSynchronize(c->stream));
            bool open = false;
            for (u32 i = 0; i < P; ++i) {
                u64 tot = 0;
                for (u32 r = 0; r < W; ++r) tot += h_all[(size_t)r * P + i];
                if (tot >= need[i]) hi[i] = mid[i]; else lo[i] = mid[i] + 1;
                open |= lo[i] < hi[i];
            }
            if (!open) round = 63;             // converged everywhere: go to the final round
        }
    }
    cut[0] = 0; cut[R] = n_local;
    for (u32 p = 1; p <= R; ++p) cut[p] = std::max(cut[p], cut[p - 1]);
    // 3. segment sizes of every rank for every partition
    std::vector<u64> seg(R);
    for (u32 p = 0; p < R; ++p) seg[p] = cut[p + 1] - cut[p];
    DevBuf d_seg(c), d_segall(c);
    TRY(d_seg.alloc((size_t)R * 8)); TRY(d_segall.alloc((size_t)W * R * 8));
    std::vector<u64> segall((size_t)W * R);
    CU(cudaMemcpyAsync(d_seg.p, seg.data(), (size_t)R * 8, cudaMemcpyHostToDevice, c->stream));
    NC(g_nccl.AllGather(d_seg.p, d_segall.p, R, ncclUint64, m->comm, c->stream));
    CU(cudaMemcpyAsync(segall.data(), d_segall.p, (size_t)W * R * 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    s->sort_part_rows.assign(R, 0);
    u64 n_recv = 0;
    for (u32 p = me; p < R; p += W)
        for (u32 r = 0; r < W; ++r) { s->sort_part_rows[p] += segall[(size_t)r * R + p]; n_recv += segall[(size_t)r * R + p]; }
    if (n_recv >= 0xFFFFFFFEull) return set_err(VB_ERR_TOO_LARGE, "rank %u would receive %llu rows", me, (unsigned long long)n_recv);
    // 4. one grouped send/recv: partition-major, source-rank-major at the receiver
    DevBuf rk(c), rv(c);
    TRY(rk.alloc(std::max<u64>(n_recv, 1) * 8));
    if (any_val) TRY(rv.alloc(std::max<u64>(n_recv, 1) * 8));
    DevBuf zero_v(c);
    if (any_val && !lv && n_local) { TRY(zero_v.alloc(n_local * 8)); CU(cudaMemsetAsync(zero_v.p, 0, n_local * 8, c->stream)); lv = zero_v.as<u64>(); }
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (c->profile) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, c->stream); }
    NC(g_nccl.GroupStart());
    for (u32 p = 0; p < R; ++p) {
        if (!seg[p]) continue;
        NC(g_nccl.Send(lk + cut[p], seg[p], ncclUint64, (int)(p % W), m->comm, c->stream));
        if (any_val) NC(g_nccl.Send(lv + cut[p], seg[p], ncclUint64, (int)(p % W), m->comm, c->stream));
    }
    u64 off = 0, sent = 0;
    for (u32 p = me; p < R; p += W)
        for (u32 r = 0; r < W; ++r) {
            const u64 cnt = segall[(size_t)r * R + p];
            if (!cnt) continue;
            NC(g_nccl.Recv(rk.as<u64>() + off, cnt, ncclUint64, (int)r, m->comm, c->stream));
            if (any_val) NC(g_nccl.Recv(rv.as<u64>() + off, cnt, ncclUint64, (int)r, m->comm, c->stream));
            off += cnt;
        }
    NC(g_nccl.GroupEnd());
    if (e0) {
        cudaEventRecord(e1, c->stream); cudaEventSynchronize(e1);
        float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
        s->xst.exchange_ms += ms;
        cudaEventDestroy(e0); cudaEventDestroy(e1);
    }
    for (u32 p = 0; p < R; ++p) if (p % W != me) sent += seg[p];
    s->xst.sent_rows += sent;
    s->xst.recv_rows += n_recv - [&] { u64 own = 0; for (u32 p = me; p < R; p += W) own += seg[p]; return own; }();
    s->xst.exchanges += 1;
    s->xst.kind = VB_XCHG_NCCL;
    s->imp_own_k = (u64 *)rk.release();
    s->imp_own_v = any_val ? (u64 *)rv.release() : nullptr;
    s->imp_keys = s->imp_own_k; s->imp_vals = s->imp_own_v; s->imp_n = n_recv;
    s->imported = true;
    std::lock_guard<std::mutex> gg(s->mu);
    s->exported = true;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_exchange(vb_shuf *s, int32_t mode)
{
    if (!s) return set_err(VB_ERR_INVALID, "NULL shuffle");
    vb_ctx *c = s->ctx;
    if (s->world < 2) return set_err(VB_ERR_STATE, "vb_shuffle_exchange needs vb_shuffle_set_dist(world > 1)");
    if (!c->comm) return set_err(VB_ERR_STATE, "vb_shuffle_exchange needs vb_ctx_comm_init");
    if (c->comm->world != s->world || c->comm->rank != s->rank) return set_err(VB_ERR_INVALID, "shuffle rank/world differ from the communicator's");
    if (mode < VB_XCHG_AUTO || mode > VB_XCHG_P2P) return set_err(VB_ERR_INVALID, "bad exchange mode");
    if (mode == VB_XCHG_AUTO) mode = is_group_op(s->agg) ? VB_XCHG_P2P : VB_XCHG_NCCL;
    if (mode == VB_XCHG_P2P && !is_group_op(s->agg)) return set_err(VB_ERR_UNSUPPORTED, "the fused P2P exchange is for GROUP/COGROUP shuffles");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    if (s->agg == VB_AGG_SORT) return exchange_sort_locked(s);
    return mode == VB_XCHG_P2P ? exchange_p2p_locked(s) : exchange_nccl_locked(s);
}

extern "C" int32_t vb_shuffle_exchange_stats(vb_shuf *s, vb_xstats *out)
{
    if (!s || !out) return set_err(VB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    cudaSetDevice(s->ctx->device);
    resolve_timers(s);
    *out = s->xst;
    return VB_OK;
}


// ---------------------------------------------------------------------------------------------
// lazy COGROUP + semi-join filter (CoGroupedRdd::compute + join, co_grouped_rdd.rs:206-249 / pair_rdd.rs:104-121)
// The reference cogroups both parents completely and then keeps the keys with values on both sides.  Grouping is the
// expensive part (dictionary + stable sort of every row), and an inner join only needs it for the keys that match:
// for BASELINE configs[3] that is 2 % of the rows.  So seal of a COGROUP shuffle only takes ownership of the rows;
// vb_join* first finds the matching keys (dictionary of the right keys, one probe per left row), compacts both sides
// to the matching rows (stable) and groups just those.  vb_shuffle_reduce* (the cogroup itself) groups everything.
// ---------------------------------------------------------------------------------------------
static bool lazy_cogroup_enabled()
{
    static const bool off = getenv("VEGA_B200_EAGER_COGROUP") != nullptr;
    return !off;
}

// take ownership of the gathered rows as SoA (copy when they are borrowed, in the shared arena, or AoS)
static int seal_lazy(vb_shuf *s, const Gathered &g, bool rows_are_owned_imports)
{
    vb_ctx *c = s->ctx;
    const u32 R = s->n_reduce;
    s->bucket_off.assign((size_t)R + 1, 0);
    s->val_off.assign((size_t)R + 1, 0);
    s->lz_n = g.n;
    s->lazy = true;
    if (g.n == 0) return VB_OK;
    if (rows_are_owned_imports) {                      // NCCL receive buffers: just keep them
        s->lz_keys = s->imp_own_k; s->lz_vals = s->imp_own_v;
        s->imp_own_k = s->imp_own_v = nullptr;
        return VB_OK;
    }
    if (!g.rows && g.keys == s->gath_keys && s->gath_keys) {   // gather_maps already made owned SoA copies
        s->lz_keys = s->gath_keys; s->lz_vals = s->gath_vals;
        s->gath_keys = s->gath_vals = nullptr;
        return VB_OK;
    }
    DevBuf k(c), v(c);
    TRY(k.alloc(g.n * 8));
    if (g.rows) {
        TRY(v.alloc(g.n * 8));
        KLaunch kl(s, K_MISC);
        u64 blocks = std::min<u64>((g.n + 255) / 256, (u64)c->sm_count * 8);
        aos_to_soa_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(g.rows, g.n, k.as<u64>(), v.as<u64>());
        TRY(kl.done("aos_to_soa_kernel"));
    } else {
        CU(cudaMemcpyAsync(k.p, g.keys, g.n * 8, cudaMemcpyDeviceToDevice, c->stream));
        if (g.vals) { TRY(v.alloc(g.n * 8)); CU(cudaMemcpyAsync(v.p, g.vals, g.n * 8, cudaMemcpyDeviceToDevice, c->stream)); }
    }
    s->lz_keys = (u64 *)k.release();
    s->lz_vals = (u64 *)v.release();
    return VB_OK;
}

static void free_lazy_rows(vb_shuf *s)
{
    dev_free(s->ctx, s->lz_keys); dev_free(s->ctx, s->lz_vals);
    s->lz_keys = s->lz_vals = nullptr;
}

// group everything (caller holds c->mu)
static int ensure_grouped(vb_shuf *s)
{
    if (!s->lazy) return VB_OK;
    Gathered g;
    g.keys = s->lz_keys; g.vals = s->lz_vals; g.n = s->lz_n;
    TRY(seal_group(s, g));
    CU(cudaStreamSynchronize(s->ctx->stream));
    free_lazy_rows(s);
    s->lazy = false;
    return VB_OK;
}

// match[i] = 1 iff keys[i] is in the dictionary; its slot is marked in slot_flag
__global__ void semi_probe_kernel(const u64 *__restrict__ keys, u64 n, Table t, unsigned char *__restrict__ slot_flag, unsigned char *__restrict__ match)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 st = (u64)gridDim.x * blockDim.x;
    const u64 pol = policy_evict_first();
    for (; i < n; i += st) {
        const u32 sl = table_find(t, ld_stream_u64(keys + i, pol));
        const bool hit = sl != 0xFFFFFFFFu;
        match[i] = hit ? 1 : 0;
        if (hit) slot_flag[sl] = 1;
    }
}
__global__ void mark_rows_kernel(const u32 *__restrict__ slot_of_row, u64 n, const unsigned char *__restrict__ slot_flag, unsigned char *__restrict__ match)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 st = (u64)gridDim.x * blockDim.x;
    for (; i < n; i += st) match[i] = slot_flag[slot_of_row[i]];
}

// stable compaction, 4096 rows per block: counts, scan, scatter
constexpr int CP_THREADS = 256, CP_ITEMS = 16, CP_TILE = CP_THREADS * CP_ITEMS;
__global__ void __launch_bounds__(CP_THREADS) compact_count_kernel(const unsigned char *__restrict__ match, u64 n, u64 *__restrict__ block_cnt)
{
    __shared__ u32 ws[CP_THREADS / 32];
    const u64 base = (u64)blockIdx.x * CP_TILE + (u64)threadIdx.x * CP_ITEMS;
    u32 c = 0;
#pragma unroll
    for (int i = 0; i < CP_ITEMS; ++i) c += (base + i < n) ? match[base + i] : 0;
    c = __reduce_add_sync(0xffffffffu, c);
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) { u32 t = 0; for (int w = 0; w < CP_THREADS / 32; ++w) t += ws[w]; block_cnt[blockIdx.x] = t; }
}
// this thread's CP_ITEMS flags (m) and the output index of its first flagged row
__device__ __forceinline__ u64 compact_first_out(const unsigned char *__restrict__ match, u64 n, const u64 *__restrict__ block_off, u64 base,
                                                 unsigned char (&m)[CP_ITEMS], u32 *ws)
{
    const u32 tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5;
    u32 c = 0;
#pragma unroll
    for (int i = 0; i < CP_ITEMS; ++i) { m[i] = (base + i < n) ? match[base + i] : 0; c += m[i]; }
    u32 incl = c;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= (u32)off) incl += t; }
    if (lane == 31) ws[warp] = incl;
    __syncthreads();
    u32 wbase = 0;
    for (u32 w = 0; w < warp; ++w) wbase += ws[w];
    return block_off[blockIdx.x] + wbase + incl - c;
}
__global__ void __launch_bounds__(CP_THREADS)
compact_scatter_kernel(const unsigned char *__restrict__ match, u64 n, const u64 *__restrict__ block_off, const u64 *__restrict__ keys,
                       const u64 *__restrict__ vals, u64 *__restrict__ out_keys, u64 *__restrict__ out_vals)
{
    __shared__ u32 ws[CP_THREADS / 32];
    const u64 base = (u64)blockIdx.x * CP_TILE + (u64)threadIdx.x * CP_ITEMS;
    unsigned char m[CP_ITEMS];
    u64 o = compact_first_out(match, n, block_off, base, m, ws);
#pragma unroll
    for (int i = 0; i < CP_ITEMS; ++i)
        if (m[i]) { out_keys[o] = keys[base + i]; if (out_vals) out_vals[o] = vals ? vals[base + i] : 0ull; ++o; }
}
// out[j] = id_base + i for the j-th flagged i
__global__ void __launch_bounds__(CP_THREADS)
compact_ids_kernel(const unsigned char *__restrict__ match, u64 n, const u64 *__restrict__ block_off, u32 id_base, u32 *__restrict__ out)
{
    __shared__ u32 ws[CP_THREADS / 32];
    const u64 base = (u64)blockIdx.x * CP_TILE + (u64)threadIdx.x * CP_ITEMS;
    unsigned char m[CP_ITEMS];
    u64 o = compact_first_out(match, n, block_off, base, m, ws);
#pragma unroll
    for (int i = 0; i < CP_ITEMS; ++i)
        if (m[i]) out[o++] = id_base + (u32)(base + i);
}

static int exclusive_scan_u64(vb_shuf *s, const u64 *in, u64 *out, u64 n, u64 *d_total);

// first half of a stable compaction: flagged rows per tile, scanned into tile offsets (off), and their total (m_out)
static int compact_offsets(vb_shuf *s, const unsigned char *match, u64 n, DevBuf &off, u64 *m_out)
{
    vb_ctx *c = s->ctx;
    const u64 blocks = (n + CP_TILE - 1) / CP_TILE;
    DevBuf cnt(c), tot(c);
    TRY(cnt.alloc(blocks * 8)); TRY(off.alloc(blocks * 8)); TRY(tot.alloc(8));
    {
        KLaunch kl(s, K_JOIN);
        compact_count_kernel<<<(unsigned)blocks, CP_THREADS, 0, c->stream>>>(match, n, cnt.as<u64>());
        TRY(kl.done("compact_count_kernel"));
    }
    TRY(exclusive_scan_u64(s, cnt.as<u64>(), off.as<u64>(), blocks, tot.as<u64>()));
    CU(cudaMemcpyAsync(c->h_scratch, tot.p, 8, cudaMemcpyDeviceToHost, c->stream));
    CU(cudaStreamSynchronize(c->stream));
    *m_out = *(u64 *)c->h_scratch;
    return VB_OK;
}

static int compact_rows(vb_shuf *s, const u64 *keys, const u64 *vals, u64 n, const unsigned char *match, DevBuf &ok, DevBuf &ov, u64 *m_out)
{
    vb_ctx *c = s->ctx;
    *m_out = 0;
    if (n == 0) return VB_OK;
    DevBuf off(c);
    u64 m = 0;
    TRY(compact_offsets(s, match, n, off, &m));
    *m_out = m;
    if (m == 0) return VB_OK;
    TRY(ok.alloc(m * 8));
    TRY(ov.alloc(m * 8));
    KLaunch kl(s, K_JOIN);
    compact_scatter_kernel<<<(unsigned)((n + CP_TILE - 1) / CP_TILE), CP_THREADS, 0, c->stream>>>(match, n, off.as<u64>(), keys, vals, ok.as<u64>(), ov.as<u64>());
    return kl.done("compact_scatter_kernel");
}

// the flagged indices i of [0, n), as id_base + i, in order (stable compaction)
static int compact_ids(vb_shuf *s, const unsigned char *flag, u64 n, u32 id_base, DevBuf &out, u64 *m_out)
{
    vb_ctx *c = s->ctx;
    *m_out = 0;
    if (n == 0) return VB_OK;
    DevBuf off(c);
    u64 m = 0;
    TRY(compact_offsets(s, flag, n, off, &m));
    *m_out = m;
    if (m == 0) return VB_OK;
    TRY(out.alloc(m * 4));
    KLaunch kl(s, K_JOIN);
    compact_ids_kernel<<<(unsigned)((n + CP_TILE - 1) / CP_TILE), CP_THREADS, 0, c->stream>>>(flag, n, off.as<u64>(), id_base, out.as<u32>());
    return kl.done("compact_ids_kernel");
}

static vb_shuf *make_internal_like(const vb_shuf *s)
{
    vb_shuf *t = new vb_shuf();
    t->ctx = s->ctx; t->id = s->id; t->n_map = 0; t->n_reduce = s->n_reduce;
    t->kdt = s->kdt; t->vdt = s->vdt; t->agg = s->agg; t->part = s->part; t->key_width = s->key_width;
    t->rank = 0; t->world = 1;                      // internal shuffles are device-local
    t->sealed = true;
    return t;
}

extern "C" int32_t vb_shuffle_free(vb_shuf *s);

// both sides lazy: internal (left, right) shuffles grouped over the rows whose key occurs on both sides
static int filtered_pair(vb_shuf *l, vb_shuf *r, vb_shuf **fl_out, vb_shuf **fr_out)
{
    auto it = l->filtered.find(r->uid);
    if (it != l->filtered.end()) { *fl_out = it->second.first; *fr_out = it->second.second; return VB_OK; }
    vb_ctx *c = l->ctx;
    vb_shuf *fl = make_internal_like(l), *fr = make_internal_like(r);
    auto fail = [&](int rc) { delete fl; delete fr; return rc; };
    fl->bucket_off.assign((size_t)l->n_reduce + 1, 0); fl->val_off = fl->bucket_off;
    fr->bucket_off = fl->bucket_off; fr->val_off = fl->bucket_off;
    if (l->lz_n && r->lz_n) {
        // 1. dictionary of the right keys (slot per right row)
        DevBuf ids_r(c);
        int rc = ids_r.alloc(r->lz_n * 4);
        if (rc) return fail(rc);
        std::vector<AggInput> in(1);
        in[0] = AggInput{IN_SOA, r->lz_keys, nullptr, r->lz_n, VB_DEVICE};
        void *tab = nullptr; u32 log_cap = 0; u64 n_ins = 0;
        rc = build_table(l, K_DICT, in, OPK_DICT, TX_NONE, r->hint, &tab, &log_cap, &n_ins, ids_r.as<u32>());
        if (rc) return fail(rc);
        DevBuf tab_guard(c); tab_guard.p = tab;
        const u64 cap = 1ull << log_cap;
        // 2. probe with every left row; 3. mark the right rows whose key matched
        DevBuf slot_flag(c), ml(c), mr(c);
        if ((rc = slot_flag.alloc(cap + 1 + 16)) || (rc = ml.alloc(l->lz_n)) || (rc = mr.alloc(r->lz_n))) return fail(rc);
        cudaMemsetAsync(slot_flag.p, 0, cap + 1 + 16, c->stream);
        {
            KLaunch kl(l, K_JOIN);
            const unsigned g = (unsigned)std::min<u64>((l->lz_n + 255) / 256, (u64)c->sm_count * 16);
            semi_probe_kernel<<<g, 256, 0, c->stream>>>(l->lz_keys, l->lz_n, table_at(tab, log_cap), slot_flag.as<unsigned char>(), ml.as<unsigned char>());
            if ((rc = kl.done("semi_probe_kernel"))) return fail(rc);
        }
        {
            KLaunch kl(l, K_JOIN);
            const unsigned g = (unsigned)std::min<u64>((r->lz_n + 255) / 256, (u64)c->sm_count * 16);
            mark_rows_kernel<<<g, 256, 0, c->stream>>>(ids_r.as<u32>(), r->lz_n, slot_flag.as<unsigned char>(), mr.as<unsigned char>());
            if ((rc = kl.done("mark_rows_kernel"))) return fail(rc);
        }
        // 4. stable compaction of both sides, then the ordinary cogroup of what is left
        DevBuf lk(c), lv(c), rk(c), rv(c);
        u64 m_l = 0, m_r = 0;
        if ((rc = compact_rows(l, l->lz_keys, l->lz_vals, l->lz_n, ml.as<unsigned char>(), lk, lv, &m_l))) return fail(rc);
        if ((rc = compact_rows(l, r->lz_keys, r->lz_vals, r->lz_n, mr.as<unsigned char>(), rk, rv, &m_r))) return fail(rc);
        if (m_l && m_r) {
            Gathered gl, gr;
            gl.keys = lk.as<u64>(); gl.vals = lv.as<u64>(); gl.n = m_l;
            gr.keys = rk.as<u64>(); gr.vals = rv.as<u64>(); gr.n = m_r;
            if ((rc = seal_group(fl, gl)) || (rc = seal_group(fr, gr))) {
                l->trash.push_back(fl); l->trash.push_back(fr);      // freed with l (vb_shuffle_free would re-lock the context here)
                return rc;
            }
            // kernel counters of the internal shuffles belong to the caller's statistics
            for (int k = 0; k < K_N; ++k) { l->klaunch[k] += fl->klaunch[k] + fr->klaunch[k]; }
            l->st.kernel_launches += fl->st.kernel_launches + fr->st.kernel_launches;
            l->st.table_slots = std::max<u64>(l->st.table_slots, std::max<u64>(cap, std::max(fl->st.table_slots, fr->st.table_slots)));
        }
        cudaStreamSynchronize(c->stream);
    }
    l->filtered[r->uid] = std::make_pair(fl, fr);
    *fl_out = fl; *fr_out = fr;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_seal(vb_shuf *s)
{
    if (!s) return set_err(VB_ERR_INVALID, "NULL shuffle");
    vb_ctx *c = s->ctx;
    {
        std::lock_guard<std::mutex> g(s->mu);
        if (s->freed) return set_err(VB_ERR_STATE, "seal of a freed shuffle");
        if (s->sealed) return VB_OK;
    }
    {
        std::unique_lock<std::mutex> g(s->mu);
        if (s->sealing) {           // concurrent seal: wait for the one in flight
            ++s->waiters;
            s->cv.wait(g, [&] { return !s->sealing || s->freed; });
            --s->waiters;
            s->cv.notify_all();
            if (s->sealed) return VB_OK;
            return set_err(VB_ERR_STATE, "shuffle %llu: the concurrent seal failed or the shuffle was freed", (unsigned long long)s->id);
        }
        if (s->sealed) return VB_OK;
        s->sealing = true;
    }
    int rc = VB_OK;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        cudaSetDevice(c->device);
        KLaunch call(s, -2);
        auto body = [&]() -> int {
            if (s->world == 1) {
                for (u32 m = 0; m < s->n_map; ++m)
                    if (!s->maps[m].present) return set_err(VB_ERR_STATE, "shuffle %llu sealed but map %u was never submitted", (unsigned long long)s->id, m);
                if (is_reduce_op(s->agg)) {
                    void *tab = nullptr; u32 log_cap = 0; u64 n_ins = 0;
                    TRY(merge_map_tables(s, &tab, &log_cap, &n_ins));
                    DevBuf guard(c); guard.p = tab;
                    TRY(finalize_reduce(s, tab, log_cap, n_ins));
                } else {
                    Gathered g;
                    TRY(gather_maps(s, &g));
                    if (s->agg == VB_AGG_SORT) TRY(seal_sort(s, g));
                    else if (s->agg == VB_AGG_COGROUP && lazy_cogroup_enabled()) TRY(seal_lazy(s, g, false));
                    else TRY(seal_group(s, g));
                }
            } else {
                if (!s->exported || !s->imported) return set_err(VB_ERR_STATE, "world > 1: seal needs export_prepare + import");
                if (is_reduce_op(s->agg)) {
                    void *tab = nullptr; u32 log_cap = 0; u64 n_ins = 0;
                    if (s->imp_n) {
                        std::vector<AggInput> in(1);
                        in[0] = AggInput{IN_SOA, s->imp_keys, s->imp_vals, s->imp_n, VB_DEVICE};
                        TRY(build_table(s, K_MERGE, in, merge_opk(s), TX_NONE, s->hint, &tab, &log_cap, &n_ins, nullptr));
                    }
                    DevBuf guard(c); guard.p = tab;
                    TRY(finalize_reduce(s, tab, log_cap, n_ins));
                } else if (s->agg == VB_AGG_SORT) {
                    if (s->sort_part_rows.size() != s->n_reduce) return set_err(VB_ERR_STATE, "multi-rank sort_by_key goes through vb_shuffle_exchange");
                    Gathered g;
                    g.keys = s->imp_keys; g.vals = s->imp_vals; g.n = s->imp_n;
                    TRY(seal_sort(s, g));        // the received runs are key-range disjoint per partition: one stable sort orders them all
                    s->bucket_off.assign((size_t)s->n_reduce + 1, 0);
                    for (u32 p = 0; p < s->n_reduce; ++p) s->bucket_off[p + 1] = s->bucket_off[p] + s->sort_part_rows[p];
                } else {
                    Gathered g;
                    g.keys = s->imp_keys; g.vals = s->imp_vals; g.n = s->imp_n;
                    if (s->agg == VB_AGG_COGROUP && lazy_cogroup_enabled()) TRY(seal_lazy(s, g, s->imp_keys == s->imp_own_k && s->imp_own_k));
                    else TRY(seal_group(s, g));
                }
            }
            release_inputs(s);
            CU(cudaStreamSynchronize(c->stream));
            return VB_OK;
        };
        rc = body();
        call.done("seal");
    }
    std::lock_guard<std::mutex> g(s->mu);
    if (rc == VB_OK) s->sealed = true; else s->failed = true;
    s->sealing = false;
    s->cv.notify_all();
    return rc;
}

extern "C" int32_t vb_shuffle_is_sealed(vb_shuf *s) { return s && s->sealed ? 1 : 0; }

static int wait_sealed(vb_shuf *s)
{
    std::unique_lock<std::mutex> g(s->mu);
    ++s->waiters;
    s->cv.wait(g, [&] { return s->sealed || s->failed || s->freed; });
    --s->waiters;
    const bool ok = s->sealed && !s->freed;
    const unsigned long long id = s->id;
    s->cv.notify_all();            // vb_shuffle_free waits for waiters == 0 (s may be deleted once g is released)
    g.unlock();
    if (!ok) return set_err(VB_ERR_STATE, "shuffle %llu failed or was freed before it was sealed", id);
    return VB_OK;
}

extern "C" int32_t vb_shuffle_reduce_size(vb_shuf *s, uint32_t r, uint64_t *n_keys, uint64_t *n_vals)
{
    if (!s) return set_err(VB_ERR_INVALID, "NULL shuffle");
    if (r >= s->n_reduce) return set_err(VB_ERR_INVALID, "reduce_id %u >= n_reduce %u", r, s->n_reduce);
    TRY(wait_sealed(s));
    if (s->lazy) {                                   // first cogroup materialisation: group all rows now
        std::lock_guard<std::mutex> lk(s->ctx->mu);
        CU(cudaSetDevice(s->ctx->device));
        TRY(ensure_grouped(s));
    }
    if (n_keys) *n_keys = s->bucket_off[r + 1] - s->bucket_off[r];
    if (n_vals) *n_vals = is_group_op(s->agg) ? s->val_off[r + 1] - s->val_off[r] : 0;
    return VB_OK;
}

static int copy_out(vb_shuf *s, void *dst, const void *src, size_t bytes, int dst_loc)
{
    if (!dst || !bytes) return VB_OK;
    if (!src) return set_err(VB_ERR_STATE, "result array missing");
    CU(cudaMemcpyAsync(dst, src, bytes, dst_loc == VB_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, s->ctx->stream));
    if (dst_loc == VB_HOST) s->st.d2h_bytes += bytes;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_reduce(vb_shuf *s, uint32_t r, void *out_keys, void *out_combined, uint64_t *out_offsets,
                                     void *out_vals, int32_t dst_loc)
{
    if (!s) return set_err(VB_ERR_INVALID, "NULL shuffle");
    if (r >= s->n_reduce) return set_err(VB_ERR_INVALID, "reduce_id %u >= n_reduce %u", r, s->n_reduce);
    if (dst_loc != VB_HOST && dst_loc != VB_DEVICE) return set_err(VB_ERR_INVALID, "bad dst_loc");
    TRY(wait_sealed(s));
    vb_ctx *c = s->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    TRY(ensure_grouped(s));
    const u64 b0 = s->bucket_off[r], nk = s->bucket_off[r + 1] - b0;
    TRY(copy_out(s, out_keys, s->res_keys ? s->res_keys + b0 : nullptr, nk * 8, dst_loc));
    if (is_group_op(s->agg)) {
        const u64 v0 = s->val_off[r], nv = s->val_off[r + 1] - v0;
        if (out_offsets) {
            if (nk == 0) {
                u64 zero = 0;
                CU(cudaMemcpyAsync(out_offsets, &zero, 8, dst_loc == VB_HOST ? cudaMemcpyHostToHost : cudaMemcpyHostToDevice, c->stream));
            } else {
                DevBuf tmp(c);
                TRY(tmp.alloc((nk + 1) * 8));
                KLaunch kl(s, K_MISC);
                rebase_kernel<<<(unsigned)((nk + 1 + 255) / 256), 256, 0, c->stream>>>(s->res_offs + b0, nk + 1, v0, tmp.as<u64>());
                TRY(kl.done("rebase_kernel"));
                TRY(copy_out(s, out_offsets, tmp.p, (nk + 1) * 8, dst_loc));
            }
        }
        TRY(copy_out(s, out_vals, s->res_vals ? s->res_vals + v0 : nullptr, nv * 8, dst_loc));
    } else if (out_combined && nk) {
        if (!s->res_comb && s->agg == VB_AGG_SORT) return set_err(VB_ERR_INVALID, "key-only sort has no payload");
        TRY(copy_out(s, out_combined, s->res_comb + b0, nk * 8, dst_loc));
    }
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// bincode blobs (N1)
// ---------------------------------------------------------------------------------------------
static u64 blob_bytes(const vb_shuf *s, u32 r)
{
    const u64 nk = s->bucket_off[r + 1] - s->bucket_off[r];
    if (is_group_op(s->agg)) return 8 + 16 * nk + 8 * (s->val_off[r + 1] - s->val_off[r]);
    return 8 + 16 * nk;
}

extern "C" int32_t vb_shuffle_reduce_blob_size(vb_shuf *s, uint32_t r, uint64_t *n_bytes)
{
    if (!s || !n_bytes) return set_err(VB_ERR_INVALID, "NULL argument");
    if (r >= s->n_reduce) return set_err(VB_ERR_INVALID, "reduce_id %u >= n_reduce %u", r, s->n_reduce);
    TRY(wait_sealed(s));
    if (s->lazy) {
        std::lock_guard<std::mutex> lk(s->ctx->mu);
        CU(cudaSetDevice(s->ctx->device));
        TRY(ensure_grouped(s));
    }
    *n_bytes = blob_bytes(s, r);
    return VB_OK;
}

extern "C" int32_t vb_shuffle_reduce_blob(vb_shuf *s, uint32_t r, void *out_blob, int32_t dst_loc)
{
    if (!s || !out_blob) return set_err(VB_ERR_INVALID, "NULL argument");
    if (r >= s->n_reduce) return set_err(VB_ERR_INVALID, "reduce_id %u >= n_reduce %u", r, s->n_reduce);
    if (dst_loc != VB_HOST && dst_loc != VB_DEVICE) return set_err(VB_ERR_INVALID, "bad dst_loc");
    TRY(wait_sealed(s));
    vb_ctx *c = s->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    TRY(ensure_grouped(s));
    const u64 bytes = blob_bytes(s, r);
    const u64 b0 = s->bucket_off[r], nk = s->bucket_off[r + 1] - b0;
    DevBuf tmp(c);
    u64 *dst = (u64 *)out_blob;
    if (dst_loc == VB_HOST) { TRY(tmp.alloc(bytes)); dst = tmp.as<u64>(); }
    const unsigned grid = (unsigned)std::min<u64>(std::max<u64>(1, (std::max(nk, s->val_off[r + 1] - s->val_off[r]) + 255) / 256), (u64)c->sm_count * 8);
    {
        KLaunch kl(s, K_MISC);
        if (is_group_op(s->agg)) {
            if (nk) blob_group_kernel<<<grid, 256, 0, c->stream>>>(s->res_keys + b0, s->res_offs + b0, nk, s->res_vals, dst);
            else CU(cudaMemsetAsync(dst, 0, 8, c->stream));
        } else {
            if (nk) blob_pairs_kernel<<<grid, 256, 0, c->stream>>>(s->res_keys + b0, s->res_comb ? s->res_comb + b0 : nullptr, nk, dst);
            else CU(cudaMemsetAsync(dst, 0, 8, c->stream));
        }
        TRY(kl.done("blob kernel"));
    }
    if (dst_loc == VB_HOST) TRY(copy_out(s, out_blob, dst, bytes, VB_HOST));
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}

extern "C" int32_t vb_shuffle_map_blob(vb_shuf *s, uint32_t map_id, const void *blob, uint64_t n_bytes, int32_t src_loc)
{
    if (!s || !blob) return set_err(VB_ERR_INVALID, "NULL argument");
    if (src_loc < VB_HOST || src_loc > VB_DEVICE_BORROWED) return set_err(VB_ERR_INVALID, "bad src_loc");
    if (s->agg == VB_AGG_SORT) return set_err(VB_ERR_UNSUPPORTED, "sort_by_key takes rows, not combined buckets");
    if (n_bytes < 8 || (n_bytes & 7)) return set_err(VB_ERR_INVALID, "corrupted blob: %llu bytes", (unsigned long long)n_bytes);
    vb_ctx *c = s->ctx;
    // the whole blob on the host: CPU-produced buckets arrive there anyway, and the record structure of
    // Vec<(K,Vec<V>)> is a linked list (each record's position depends on the previous lengths)
    std::vector<u64> host;
    const u64 *w = (const u64 *)blob;
    if (src_loc != VB_HOST) {
        host.resize(n_bytes / 8);
        std::lock_guard<std::mutex> lk(c->mu);
        CU(cudaSetDevice(c->device));
        CU(cudaMemcpyAsync(host.data(), blob, n_bytes, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        w = host.data();
    }
    const u64 words = n_bytes / 8, n = w[0];
    if (!is_group_op(s->agg)) {
        if (n > (words - 1) / 2 || words != 1 + 2 * n) return set_err(VB_ERR_INVALID, "corrupted blob: %llu records in %llu bytes", (unsigned long long)n, (unsigned long long)n_bytes);
        std::vector<u64> k(n), v(n);
        for (u64 i = 0; i < n; ++i) { k[i] = w[1 + 2 * i]; v[i] = w[2 + 2 * i]; }
        return shuffle_map(s, map_id, nullptr, k.data(), v.data(), n, VB_HOST, /*combined=*/true);
    }
    std::vector<u64> k, v;
    u64 pos = 1;
    for (u64 i = 0; i < n; ++i) {
        if (pos + 2 > words) return set_err(VB_ERR_INVALID, "corrupted blob: record %llu runs past the end", (unsigned long long)i);
        const u64 key = w[pos], len = w[pos + 1];
        if (len > words - pos - 2) return set_err(VB_ERR_INVALID, "corrupted blob: record %llu has length %llu", (unsigned long long)i, (unsigned long long)len);
        for (u64 j = 0; j < len; ++j) { k.push_back(key); v.push_back(w[pos + 2 + j]); }
        pos += 2 + len;
    }
    if (pos != words) return set_err(VB_ERR_INVALID, "corrupted blob: %llu trailing bytes", (unsigned long long)((words - pos) * 8));
    return shuffle_map(s, map_id, nullptr, k.data(), v.data(), k.size(), VB_HOST, false);
}

// ---------------------------------------------------------------------------------------------
// join
// ---------------------------------------------------------------------------------------------
static int exclusive_scan_u64(vb_shuf *s, const u64 *in, u64 *out, u64 n, u64 *d_total)
{
    vb_ctx *c = s->ctx;
    if (n == 0) return VB_OK;
    const u64 blocks = (n + SC_CHUNK - 1) / SC_CHUNK;
    if (blocks == 1) {
        KLaunch kl(s, K_JOIN);
        scan_apply_kernel<<<1, SC_THREADS, 0, c->stream>>>(in, out, n, nullptr, d_total);
        return kl.done("scan_apply_kernel");
    }
    DevBuf sums(c), offs(c);
    TRY(sums.alloc(blocks * 8));
    TRY(offs.alloc(blocks * 8));
    {
        KLaunch kl(s, K_JOIN);
        scan_reduce_kernel<<<(unsigned)blocks, SC_THREADS, 0, c->stream>>>(in, n, sums.as<u64>());
        TRY(kl.done("scan_reduce_kernel"));
    }
    TRY(exclusive_scan_u64(s, sums.as<u64>(), offs.as<u64>(), blocks, nullptr));
    KLaunch kl(s, K_JOIN);
    scan_apply_kernel<<<(unsigned)blocks, SC_THREADS, 0, c->stream>>>(in, out, n, offs.as<u64>(), d_total);
    return kl.done("scan_apply_kernel");
}

static int join_check(vb_shuf *l, vb_shuf *r, u32 rid)
{
    if (!l || !r) return set_err(VB_ERR_INVALID, "NULL shuffle");
    if (!is_group_op(l->agg) || !is_group_op(r->agg)) return set_err(VB_ERR_INVALID, "join needs two GROUP/COGROUP shuffles");
    if (l->n_reduce != r->n_reduce || l->key_width != r->key_width) return set_err(VB_ERR_INVALID, "join sides use different partitioners");
    if (l->ctx != r->ctx) return set_err(VB_ERR_INVALID, "join sides live on different contexts");
    if (rid >= l->n_reduce) return set_err(VB_ERR_INVALID, "reduce_id %u >= n_reduce %u", rid, l->n_reduce);
    TRY(wait_sealed(l));
    TRY(wait_sealed(r));
    return VB_OK;
}

static int join_plan(vb_shuf *l, vb_shuf *r, u32 rid, JoinPlan **out)
{
    vb_ctx *c = l->ctx;
    auto key = std::make_pair((const vb_shuf *)r, rid);
    auto it = l->join_plans.find(key);
    if (it != l->join_plans.end()) { *out = &it->second; return VB_OK; }
    JoinPlan p;
    const u64 lb = l->bucket_off[rid], le = l->bucket_off[rid + 1];
    p.nl = (u32)(le - lb);
    if (p.nl && r->n_keys && r->dict) {
        DevBuf cnt(c), pos(c), match(c), tot(c);
        TRY(cnt.alloc((u64)p.nl * 8));
        TRY(pos.alloc((u64)p.nl * 8));
        TRY(match.alloc((u64)p.nl * 4));
        TRY(tot.alloc(8));
        {
            KLaunch kl(l, K_JOIN);
            join_probe_kernel<<<(p.nl + 255) / 256, 256, 0, c->stream>>>(l->res_keys, l->res_offs, (u32)lb, (u32)le,
                                                                         table_at(r->dict, r->dict_log_cap), r->dense_of_slot,
                                                                         r->res_offs, cnt.as<u64>(), match.as<u32>());
            TRY(kl.done("join_probe_kernel"));
        }
        TRY(exclusive_scan_u64(l, cnt.as<u64>(), pos.as<u64>(), p.nl, tot.as<u64>()));
        CU(cudaMemcpyAsync(c->h_scratch, tot.p, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        p.total = *(u64 *)c->h_scratch;
        p.pos = (u64 *)pos.release();
        p.match = (u32 *)match.release();
    }
    auto ins = l->join_plans.emplace(key, p);
    *out = &ins.first->second;
    return VB_OK;
}

// the pair of shuffles whose CSR the join reads: the filtered internal pair while both sides are still lazy
static int join_sides(vb_shuf *&l, vb_shuf *&r)
{
    if (l->lazy && r->lazy && l != r) {
        vb_shuf *fl = nullptr, *fr = nullptr;
        TRY(filtered_pair(l, r, &fl, &fr));
        l = fl; r = fr;
        return VB_OK;
    }
    TRY(ensure_grouped(l));
    TRY(ensure_grouped(r));
    return VB_OK;
}

extern "C" int32_t vb_join_size(vb_shuf *l, vb_shuf *r, uint32_t rid, uint64_t *n_out)
{
    TRY(join_check(l, r, rid));
    if (!n_out) return set_err(VB_ERR_INVALID, "n_out is NULL");
    std::lock_guard<std::mutex> lk(l->ctx->mu);
    CU(cudaSetDevice(l->ctx->device));
    TRY(join_sides(l, r));
    JoinPlan *p = nullptr;
    TRY(join_plan(l, r, rid, &p));
    *n_out = p->total;
    return VB_OK;
}

extern "C" int32_t vb_join(vb_shuf *l, vb_shuf *r, uint32_t rid, void *out_k, void *out_v, void *out_w, int32_t dst_loc)
{
    TRY(join_check(l, r, rid));
    if (dst_loc != VB_HOST && dst_loc != VB_DEVICE) return set_err(VB_ERR_INVALID, "bad dst_loc");
    vb_ctx *c = l->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    TRY(join_sides(l, r));
    JoinPlan *p = nullptr;
    TRY(join_plan(l, r, rid, &p));
    const u64 total = p->total;
    int rc = VB_OK;
    if (total) {
        if (!out_k || !out_v || !out_w) return set_err(VB_ERR_INVALID, "NULL output with %llu rows to write", (unsigned long long)total);
        DevBuf bk(c), bv(c), bw(c);
        u64 *dk = (u64 *)out_k, *dv = (u64 *)out_v, *dw = (u64 *)out_w;
        if (dst_loc == VB_HOST) {
            TRY(bk.alloc(total * 8)); TRY(bv.alloc(total * 8)); TRY(bw.alloc(total * 8));
            dk = bk.as<u64>(); dv = bv.as<u64>(); dw = bw.as<u64>();
        }
        {
            KLaunch kl(l, K_JOIN);
            u64 blocks = std::min<u64>((total + 255) / 256, (u64)c->sm_count * 8);
            join_expand_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(p->pos, p->nl, total, l->res_keys, l->res_offs, l->res_vals,
                                                                        (u32)l->bucket_off[rid], p->match, r->res_offs, r->res_vals,
                                                                        dk, dv, dw);
            rc = kl.done("join_expand_kernel");
        }
        if (rc == VB_OK && dst_loc == VB_HOST) {
            rc = copy_out(l, out_k, dk, total * 8, VB_HOST);
            if (rc == VB_OK) rc = copy_out(l, out_v, dv, total * 8, VB_HOST);
            if (rc == VB_OK) rc = copy_out(l, out_w, dw, total * 8, VB_HOST);
        }
        cudaStreamSynchronize(c->stream);
    }
    dev_free(c, p->pos);
    dev_free(c, p->match);
    l->join_plans.erase(std::make_pair((const vb_shuf *)r, rid));
    return rc;
}

// ---------------------------------------------------------------------------------------------
// cogroup and outer joins (PairRdd::cogroup, pair_rdd.rs:123-155 / co_grouped_rdd.rs:206-249; the outer joins are
// Spark's).  Both need every key of a side, so both sides are grouped completely (no semi-join filter).  Per
// partition: probe the right dictionary with the left keys (match + "seen" flags), compact the unseen right keys,
// then either lay out both value lists in union order (cogroup) or expand the rows an outer join keeps.
// ---------------------------------------------------------------------------------------------
static void free_cogroup_plan(vb_ctx *c, CogroupPlan &p)
{
    dev_free(c, p.match); dev_free(c, p.ronly); dev_free(c, p.rowpos);
    p = CogroupPlan();
}

static int cogroup_plan(vb_shuf *l, vb_shuf *r, u32 rid, CogroupPlan **out)
{
    vb_ctx *c = l->ctx;
    const auto key = std::make_pair(r->uid, rid);
    auto it = l->cg_plans.find(key);
    if (it != l->cg_plans.end()) { *out = &it->second; return VB_OK; }
    const u64 lb = l->bucket_off[rid], rb = r->bucket_off[rid];
    const u32 nl = (u32)(l->bucket_off[rid + 1] - lb), nr = (u32)(r->bucket_off[rid + 1] - rb);
    DevBuf match(c), ronly(c);
    u64 nro = 0;
    if (nl) {
        TRY(match.alloc((u64)nl * 4));
        if (!nr) CU(cudaMemsetAsync(match.p, 0xFF, (u64)nl * 4, c->stream));
    }
    if (nr) {
        DevBuf flag(c);
        TRY(flag.alloc(nr));
        CU(cudaMemsetAsync(flag.p, 1, nr, c->stream));
        if (nl) {
            KLaunch kl(l, K_JOIN);
            cogroup_probe_kernel<<<(nl + 255) / 256, 256, 0, c->stream>>>(l->res_keys, (u32)lb, nl, table_at(r->dict, r->dict_log_cap),
                                                                           r->dense_of_slot, (u32)rb, (u32)rb + nr, match.as<u32>(),
                                                                           flag.as<unsigned char>());
            TRY(kl.done("cogroup_probe_kernel"));
        }
        TRY(compact_ids(l, flag.as<unsigned char>(), nr, (u32)rb, ronly, &nro));
    }
    CogroupPlan p;
    p.nl = nl;
    p.nro = (u32)nro;
    p.match = (u32 *)match.release();
    p.ronly = (u32 *)ronly.release();
    *out = &l->cg_plans.emplace(key, p).first->second;
    return VB_OK;
}

// row positions of an outer join of `kind` over the plan's union keys (cached for the fetch that follows a size call)
static int cogroup_rows(vb_shuf *l, vb_shuf *r, u32 rid, CogroupPlan *p, int kind)
{
    if (p->kind == kind) return VB_OK;
    vb_ctx *c = l->ctx;
    dev_free(c, p->rowpos);
    p->rowpos = nullptr;
    p->rows = 0;
    p->kind = 0;
    const u32 nu = p->nl + p->nro;
    if (nu) {
        DevBuf cnt(c), pos(c), tot(c);
        TRY(cnt.alloc((u64)nu * 8)); TRY(pos.alloc((u64)nu * 8)); TRY(tot.alloc(8));
        {
            KLaunch kl(l, K_JOIN);
            cogroup_count_kernel<<<(nu + 255) / 256, 256, 0, c->stream>>>(p->nl, nu, (u32)l->bucket_off[rid], l->res_offs, p->match, p->ronly,
                                                                          r->res_offs, kind, nullptr, nullptr, cnt.as<u64>());
            TRY(kl.done("cogroup_count_kernel"));
        }
        TRY(exclusive_scan_u64(l, cnt.as<u64>(), pos.as<u64>(), nu, tot.as<u64>()));
        CU(cudaMemcpyAsync(c->h_scratch, tot.p, 8, cudaMemcpyDeviceToHost, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        p->rows = *(u64 *)c->h_scratch;
        p->rowpos = (u64 *)pos.release();
    }
    p->kind = kind;
    return VB_OK;
}

// both sides grouped completely (caller holds c->mu)
static int cogroup_sides(vb_shuf *l, vb_shuf *r)
{
    TRY(ensure_grouped(l));
    return ensure_grouped(r);
}

static void drop_cogroup_plan(vb_shuf *l, vb_shuf *r, u32 rid)
{
    auto it = l->cg_plans.find(std::make_pair(r->uid, rid));
    if (it == l->cg_plans.end()) return;
    free_cogroup_plan(l->ctx, it->second);
    l->cg_plans.erase(it);
}

extern "C" int32_t vb_cogroup_size(vb_shuf *l, vb_shuf *r, uint32_t rid, uint64_t *n_keys, uint64_t *n_left_vals, uint64_t *n_right_vals)
{
    TRY(join_check(l, r, rid));
    std::lock_guard<std::mutex> lk(l->ctx->mu);
    CU(cudaSetDevice(l->ctx->device));
    TRY(cogroup_sides(l, r));
    CogroupPlan *p = nullptr;
    TRY(cogroup_plan(l, r, rid, &p));
    if (n_keys) *n_keys = (u64)p->nl + p->nro;
    if (n_left_vals) *n_left_vals = l->val_off[rid + 1] - l->val_off[rid];
    if (n_right_vals) *n_right_vals = r->val_off[rid + 1] - r->val_off[rid];
    return VB_OK;
}

// the caller's buffer when it is device memory, else a temporary device buffer copied out at the end
static int cogroup_target(vb_ctx *c, void *dst, int dst_loc, DevBuf &tmp, u64 bytes, void **out)
{
    if (dst_loc == VB_DEVICE) { *out = dst; return VB_OK; }
    TRY(tmp.alloc(bytes));
    *out = tmp.p;
    return VB_OK;
}

static int cogroup_fetch(vb_shuf *l, vb_shuf *r, u32 rid, const CogroupPlan *p, void *out_keys, uint64_t *out_offs_l, void *out_vals_l,
                         uint64_t *out_offs_r, void *out_vals_r, int32_t dst_loc)
{
    vb_ctx *c = l->ctx;
    const u32 nl = p->nl, nu = p->nl + p->nro;
    const u64 lb = l->bucket_off[rid];
    const u64 lv0 = l->val_off[rid], nlv = l->val_off[rid + 1] - lv0;
    const u64 nrv = r->val_off[rid + 1] - r->val_off[rid];
    if (nu == 0) {
        const u64 zero = 0;
        for (uint64_t *o : {out_offs_l, out_offs_r})
            if (o) CU(cudaMemcpyAsync(o, &zero, 8, dst_loc == VB_HOST ? cudaMemcpyHostToHost : cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        return VB_OK;
    }
    if (!out_keys || !out_offs_l || !out_offs_r || (nlv && !out_vals_l) || (nrv && !out_vals_r))
        return set_err(VB_ERR_INVALID, "NULL output with %u keys to write", nu);
    DevBuf cl(c), cr(c), bk(c), bol(c), bor(c), bvr(c);
    void *dk = nullptr, *dol = nullptr, *dor = nullptr, *dvr = nullptr;
    TRY(cogroup_target(c, out_keys, dst_loc, bk, (u64)nu * 8, &dk));
    TRY(cogroup_target(c, out_offs_l, dst_loc, bol, ((u64)nu + 1) * 8, &dol));
    TRY(cogroup_target(c, out_offs_r, dst_loc, bor, ((u64)nu + 1) * 8, &dor));
    TRY(cogroup_target(c, out_vals_r, dst_loc, bvr, nrv * 8, &dvr));
    // value counts per union key, scanned into the two offset arrays (offs[nu] = the side's value count)
    TRY(cl.alloc((u64)nu * 8)); TRY(cr.alloc((u64)nu * 8));
    {
        KLaunch kl(l, K_JOIN);
        cogroup_count_kernel<<<(nu + 255) / 256, 256, 0, c->stream>>>(nl, nu, (u32)lb, l->res_offs, p->match, p->ronly, r->res_offs, 0,
                                                                      cl.as<u64>(), cr.as<u64>(), nullptr);
        TRY(kl.done("cogroup_count_kernel"));
    }
    TRY(exclusive_scan_u64(l, cl.as<u64>(), (u64 *)dol, nu, (u64 *)dol + nu));
    TRY(exclusive_scan_u64(l, cr.as<u64>(), (u64 *)dor, nu, (u64 *)dor + nu));
    // union keys: the left key slice, then the right-only keys
    if (nl) CU(cudaMemcpyAsync(dk, l->res_keys + lb, (u64)nl * 8, cudaMemcpyDeviceToDevice, c->stream));
    if (p->nro) {
        KLaunch kl(l, K_JOIN);
        cogroup_keys_kernel<<<(p->nro + 255) / 256, 256, 0, c->stream>>>(p->ronly, p->nro, r->res_keys, (u64 *)dk + nl);
        TRY(kl.done("cogroup_keys_kernel"));
    }
    // right values: segmented gather in union order
    if (nrv) {
        KLaunch kl(l, K_JOIN);
        const u64 blocks = std::min<u64>((nrv + 255) / 256, (u64)c->sm_count * 8);
        cogroup_gather_right_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>((const u64 *)dor, nu, nrv, nl, p->match, p->ronly, r->res_offs,
                                                                             r->res_vals, (u64 *)dvr);
        TRY(kl.done("cogroup_gather_right_kernel"));
    }
    // left values: the partition's left CSR is already in union order
    TRY(copy_out(l, out_vals_l, l->res_vals ? l->res_vals + lv0 : nullptr, nlv * 8, dst_loc));
    if (dst_loc == VB_HOST) {
        TRY(copy_out(l, out_keys, dk, (u64)nu * 8, VB_HOST));
        TRY(copy_out(l, out_offs_l, dol, ((u64)nu + 1) * 8, VB_HOST));
        TRY(copy_out(l, out_offs_r, dor, ((u64)nu + 1) * 8, VB_HOST));
        TRY(copy_out(l, out_vals_r, dvr, nrv * 8, VB_HOST));
    }
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}

extern "C" int32_t vb_cogroup(vb_shuf *l, vb_shuf *r, uint32_t rid, void *out_keys, uint64_t *out_offs_l, void *out_vals_l,
                              uint64_t *out_offs_r, void *out_vals_r, int32_t dst_loc)
{
    TRY(join_check(l, r, rid));
    if (dst_loc != VB_HOST && dst_loc != VB_DEVICE) return set_err(VB_ERR_INVALID, "bad dst_loc");
    vb_ctx *c = l->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    TRY(cogroup_sides(l, r));
    CogroupPlan *p = nullptr;
    TRY(cogroup_plan(l, r, rid, &p));
    const int rc = cogroup_fetch(l, r, rid, p, out_keys, out_offs_l, out_vals_l, out_offs_r, out_vals_r, dst_loc);
    cudaStreamSynchronize(c->stream);
    drop_cogroup_plan(l, r, rid);
    return rc;
}

static bool outer_kind_ok(int32_t kind) { return kind == VB_JOIN_LEFT_OUTER || kind == VB_JOIN_RIGHT_OUTER || kind == VB_JOIN_FULL_OUTER; }

extern "C" int32_t vb_join_outer_size(vb_shuf *l, vb_shuf *r, uint32_t rid, int32_t kind, uint64_t *n_out)
{
    TRY(join_check(l, r, rid));
    if (!outer_kind_ok(kind)) return set_err(VB_ERR_INVALID, "bad outer join kind %d", kind);
    if (!n_out) return set_err(VB_ERR_INVALID, "n_out is NULL");
    std::lock_guard<std::mutex> lk(l->ctx->mu);
    CU(cudaSetDevice(l->ctx->device));
    TRY(cogroup_sides(l, r));
    CogroupPlan *p = nullptr;
    TRY(cogroup_plan(l, r, rid, &p));
    TRY(cogroup_rows(l, r, rid, p, kind));
    *n_out = p->rows;
    return VB_OK;
}

extern "C" int32_t vb_join_outer(vb_shuf *l, vb_shuf *r, uint32_t rid, int32_t kind, void *out_k, void *out_v, void *out_w,
                                 uint8_t *out_valid, int32_t dst_loc)
{
    TRY(join_check(l, r, rid));
    if (!outer_kind_ok(kind)) return set_err(VB_ERR_INVALID, "bad outer join kind %d", kind);
    if (dst_loc != VB_HOST && dst_loc != VB_DEVICE) return set_err(VB_ERR_INVALID, "bad dst_loc");
    vb_ctx *c = l->ctx;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    TRY(cogroup_sides(l, r));
    CogroupPlan *p = nullptr;
    TRY(cogroup_plan(l, r, rid, &p));
    int rc = cogroup_rows(l, r, rid, p, kind);
    const u64 total = p->rows;
    if (rc == VB_OK && total) {
        if (!out_k || !out_v || !out_w) rc = set_err(VB_ERR_INVALID, "NULL output with %llu rows to write", (unsigned long long)total);
        DevBuf bk(c), bv(c), bw(c), bvalid(c);
        void *dk = nullptr, *dv = nullptr, *dw = nullptr, *dvalid = nullptr;
        if (rc == VB_OK) rc = cogroup_target(c, out_k, dst_loc, bk, total * 8, &dk);
        if (rc == VB_OK) rc = cogroup_target(c, out_v, dst_loc, bv, total * 8, &dv);
        if (rc == VB_OK) rc = cogroup_target(c, out_w, dst_loc, bw, total * 8, &dw);
        if (rc == VB_OK && out_valid) rc = cogroup_target(c, out_valid, dst_loc, bvalid, total, &dvalid);
        if (rc == VB_OK) {
            KLaunch kl(l, K_JOIN);
            const u64 blocks = std::min<u64>((total + 255) / 256, (u64)c->sm_count * 8);
            outer_expand_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(p->rowpos, p->nl + p->nro, total, p->nl, (u32)l->bucket_off[rid],
                                                                         l->res_keys, l->res_offs, l->res_vals, p->match, p->ronly,
                                                                         r->res_keys, r->res_offs, r->res_vals, (u64 *)dk, (u64 *)dv,
                                                                         (u64 *)dw, (unsigned char *)dvalid);
            rc = kl.done("outer_expand_kernel");
        }
        if (rc == VB_OK && dst_loc == VB_HOST) {
            rc = copy_out(l, out_k, dk, total * 8, VB_HOST);
            if (rc == VB_OK) rc = copy_out(l, out_v, dv, total * 8, VB_HOST);
            if (rc == VB_OK) rc = copy_out(l, out_w, dw, total * 8, VB_HOST);
            if (rc == VB_OK && out_valid) rc = copy_out(l, out_valid, dvalid, total, VB_HOST);
        }
        cudaStreamSynchronize(c->stream);
    }
    drop_cogroup_plan(l, r, rid);
    return rc;
}

// ---------------------------------------------------------------------------------------------
// free / stats
// ---------------------------------------------------------------------------------------------
extern "C" int32_t vb_shuffle_free(vb_shuf *s)
{
    if (!s) return VB_OK;
    vb_ctx *c = s->ctx;
    {
        std::unique_lock<std::mutex> g(s->mu);
        s->freed = true;
        s->cv.notify_all();
        s->cv.wait(g, [&] { return s->waiters == 0 && !s->sealing; });   // blocked reduce/join/seal callers leave first
    }
    {
        std::lock_guard<std::mutex> lk(c->mu);
        cudaSetDevice(c->device);
        resolve_timers(s);
        for (auto &m : s->maps) free_map(s, m);
        release_inputs(s);
        dev_free(c, s->res_keys); dev_free(c, s->res_comb); dev_free(c, s->res_offs); dev_free(c, s->res_vals);
        dev_free(c, s->dict); dev_free(c, s->dense_of_slot);
        for (auto &kv : s->join_plans) { dev_free(c, kv.second.pos); dev_free(c, kv.second.match); }
        for (auto &kv : s->cg_plans) free_cogroup_plan(c, kv.second);
        free_lazy_rows(s);
        cudaStreamSynchronize(c->stream);
    }
    for (auto &kv : s->filtered) { vb_shuffle_free(kv.second.first); vb_shuffle_free(kv.second.second); }
    for (vb_shuf *t : s->trash) vb_shuffle_free(t);
    delete s;
    return VB_OK;
}

extern "C" int32_t vb_shuffle_stats(vb_shuf *s, vb_stats *out)
{
    if (!s || !out) return set_err(VB_ERR_INVALID, "NULL argument");
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    cudaSetDevice(s->ctx->device);
    resolve_timers(s);
    *out = s->st;
    return VB_OK;
}

// per-kernel-class device time (profiling on): klass 0 hash_agg, 1 dict, 2 merge, 3 rp_hist,
// 4 rp_scan, 5 rp_scatter, 6 misc, 7 join
extern "C" int32_t vb_shuffle_kernel_time(vb_shuf *s, int32_t klass, double *ms, uint64_t *launches)
{
    if (!s || klass < 0 || klass >= K_N) return set_err(VB_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(s->ctx->mu);
    cudaSetDevice(s->ctx->device);
    resolve_timers(s);
    if (ms) *ms = s->kms[klass];
    if (launches) *launches = s->klaunch[klass];
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// host-side pieces of the path
// ---------------------------------------------------------------------------------------------
extern "C" uint64_t vb_hash_key(uint64_t key, uint32_t key_width) { return hash_key(key, key_width); }

extern "C" uint32_t vb_get_partition(uint64_t key, uint32_t key_width, uint32_t n_reduce)
{
    if (n_reduce == 0) return 0;
    return (uint32_t)(hash_key(key, key_width) % (uint64_t)n_reduce);
}

// ParallelCollection::slice (src/rdd/parallel_collection_rdd.rs:116-145).  The reference walks the
// elements and cuts at most once per element; in closed form that is
//   n >= num_slices : exactly num_slices slices, slice s = [floor(s*n/num_slices), floor((s+1)*n/num_slices))
//   n <  num_slices : every element triggers a cut (the running `end` never gets ahead of the element
//                     index), giving an empty leading slice followed by n singletons (n+1 slices)
// (tests/test_abi_cpu.py checks this against the literal loop of the oracle).
extern "C" uint64_t vb_slice(uint64_t n, uint64_t num_slices, uint64_t *starts)
{
    if (num_slices < 1 || !starts) return 0;
    if (n >= num_slices) {
        for (uint64_t s = 0; s < num_slices; ++s) starts[s] = (uint64_t)(((unsigned __int128)s * n) / num_slices);
        starts[num_slices] = n;
        return num_slices;
    }
    starts[0] = 0;
    for (uint64_t i = 0; i < n; ++i) starts[i + 1] = i;
    starts[n + 1] = n;
    return n + 1;
}

// ---------------------------------------------------------------------------------------------
// device-resident sources
// ---------------------------------------------------------------------------------------------
__global__ void range_kernel(u64 *__restrict__ out, u64 start, u64 step, u64 n)
{
    u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x;
    const u64 st = (u64)gridDim.x * blockDim.x;
    for (; i < n; i += st) out[i] = start + i * step;
}

// Context::range (src/context.rs:419-431): the elements of (start..=end).step_by(step), written on the device.
extern "C" uint64_t vb_range_len(uint64_t start, uint64_t end, uint64_t step)
{
    if (step == 0 || end < start) return 0;
    return (end - start) / step + 1;
}

extern "C" int32_t vb_range(vb_ctx *c, void *out_dev, uint64_t start, uint64_t end, uint64_t step)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    if (step == 0) return set_err(VB_ERR_INVALID, "step must be >= 1 (Rust's step_by panics on 0)");
    const u64 n = vb_range_len(start, end, step);
    if (n == 0) return VB_OK;
    if (!out_dev) return set_err(VB_ERR_INVALID, "out_dev is NULL");
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    const u64 blocks = std::min<u64>((n + 255) / 256, (u64)c->sm_count * 16);
    range_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>((u64 *)out_dev, start, step, n);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}

// ---------------------------------------------------------------------------------------------
// synthetic input
// ---------------------------------------------------------------------------------------------
extern "C" int32_t vb_gen_pairs(vb_ctx *c, void *rows_dev, void *keys_dev, void *vals_dev, uint64_t first, uint64_t n,
                                int32_t mode, uint64_t n_distinct, uint64_t rank_base, uint64_t seed_k, uint64_t seed_v,
                                double zipf_s)
{
    if (!c) return set_err(VB_ERR_INVALID, "ctx is NULL");
    if (!rows_dev && !keys_dev) return set_err(VB_ERR_INVALID, "no output buffer");
    if (mode < GEN_UNIFORM || mode > GEN_UNIQUE) return set_err(VB_ERR_INVALID, "bad generator mode");
    if (mode != GEN_UNIQUE && n_distinct == 0) return set_err(VB_ERR_INVALID, "n_distinct must be > 0");
    if (n == 0) return VB_OK;
    std::lock_guard<std::mutex> lk(c->mu);
    CU(cudaSetDevice(c->device));
    if (mode == GEN_ZIPF && (c->zipf_n != n_distinct || c->zipf_s != zipf_s)) {
        std::vector<double> cdf(n_distinct);
        long double h = 0;
        for (u64 k = 0; k < n_distinct; ++k) { h += 1.0L / powl((long double)(k + 1), (long double)zipf_s); cdf[k] = (double)h; }
        for (u64 k = 0; k < n_distinct; ++k) cdf[k] = (double)(cdf[k] / (double)h);
        cdf[n_distinct - 1] = 1.0;
        if (c->zipf_cdf) cudaFreeAsync(c->zipf_cdf, c->stream);
        c->zipf_cdf = nullptr;
        CU(cudaMallocAsync((void **)&c->zipf_cdf, n_distinct * 8, c->pool, c->stream));
        CU(cudaMemcpyAsync(c->zipf_cdf, cdf.data(), n_distinct * 8, cudaMemcpyHostToDevice, c->stream));
        CU(cudaStreamSynchronize(c->stream));
        c->zipf_n = n_distinct;
        c->zipf_s = zipf_s;
    }
    u64 blocks = std::min<u64>((n + 255) / 256, (u64)c->sm_count * 16);
    gen_pairs_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>((u64 *)rows_dev, (u64 *)keys_dev, (u64 *)vals_dev, first, n, mode,
                                                              n_distinct, rank_base, seed_k, seed_v, c->zipf_cdf);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(c->stream));
    return VB_OK;
}
