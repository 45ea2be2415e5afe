// splendor_b200.cu -- C-ABI entry points (include/splendor_b200.h) and the native host driver of
// the level-synchronous search.  Build: nvcc -gencode arch=compute_100a,code=sm_100a (see
// __graft_entry__.build()).  No CPU fallback: without a usable device every compute call fails.
#include "../../include/splendor_b200.h"

#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "spl_kernels.cuh"
#include "spl_m2.cuh"
#include "spl_shard.cuh"
#include "spl_realistic.cuh"
#include "spl_sbatch.cuh"
#include "spl_tables.cuh"

using namespace spl;

// parents per round of a level (spl_config.chunk_parents is clamped to it); a grouped round numbers its parents in the
// ITEM_PARENT_BITS of a buy's sort item
constexpr uint64_t MAX_CHUNK_PARENTS = 16ull << 20;
static_assert(MAX_CHUNK_PARENTS <= (1ull << ITEM_PARENT_BITS), "a round's parent index must fit the item of its buys");

static std::string g_create_error;

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    ~DevBuf() { release(); }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    // grow to at least `bytes` (geometric), optionally preserving the first `keep` bytes
    cudaError_t ensure(size_t bytes, size_t keep, cudaStream_t st) {
        if (bytes <= cap) return cudaSuccess;
        size_t ncap = std::max(bytes, cap + cap / 2);
        ncap = (ncap + 255) & ~(size_t)255;
        void *np = nullptr;
        cudaError_t e = cudaMalloc(&np, ncap);
        if (e != cudaSuccess && ncap > bytes) {  // retry with the exact size
            cudaGetLastError();
            ncap = (bytes + 255) & ~(size_t)255;
            e = cudaMalloc(&np, ncap);
        }
        if (e != cudaSuccess) return e;
        if (keep && p) {
            e = cudaMemcpyAsync(np, p, keep, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) { cudaFree(np); return e; }
        }
        if (p) cudaFree(p);
        p = np;
        cap = ncap;
        return cudaSuccess;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
    void swap(DevBuf &o) { std::swap(p, o.p); std::swap(cap, o.cap); }
};

static inline unsigned nblk(int64_t n, int per = TILE) { return (unsigned)((n + per - 1) / per); }

// The key table is sized in slots (3 per 64-byte bucket); slot ids are u32 (bucket << 2 | slot), so at most 2^30 buckets.
constexpr uint64_t MAX_BUCKETS = 1ull << 30;
static uint64_t buckets_for(uint64_t slots) {
    return std::min<uint64_t>(std::max<uint64_t>(slots / BUCKET_SLOTS, 16), MAX_BUCKETS);
}

// What differs between the three visited tables: their unit, how full they may get, and their rehash kernel.
struct TableDesc {
    uint64_t unit_bytes, unit_slots, max_units;  // a unit (bucket or card-set node): its bytes and its entry slots
    double load;                                 // grow while entries + need > load * slots ...
    uint64_t full_div;                           // ... and fail if then entries + need / full_div > slots - slots / 16
    void (*rehash)(const void *from, uint64_t units, void *to, uint64_t to_units, Counters *ctr, cudaStream_t st);
    const char *rehash_msg;                      // %llu: the new number of units
    const char *full_msg;                        // %llu x 4: entries, need, slots, byte ceiling
};
static const TableDesc KEY_TABLE_DESC = {
    64, BUCKET_SLOTS, MAX_BUCKETS, 0.7, 8,
    [](const void *from, uint64_t units, void *to, uint64_t to_units, Counters *ctr, cudaStream_t st) {
        rehash_kernel<<<nblk((int64_t)(units * BUCKET_SLOTS)), TILE, 0, st>>>(static_cast<const uint64_t *>(from), units,
                                                                              static_cast<uint64_t *>(to), to_units, ctr);
    },
    "rehash into %llu buckets overflowed a probe sequence",
    "visited table full: %llu occupied + %llu candidates vs %llu slots (max_table_bytes=%llu)"};
static const TableDesc NODE_TABLE_DESC = {
    NODE_WORDS * 8, 1, ~0ull, 0.6, 1,
    [](const void *from, uint64_t units, void *to, uint64_t to_units, Counters *ctr, cudaStream_t st) {
        m2_rehash_kernel<<<nblk((int64_t)units * 32), TILE, 0, st>>>(static_cast<const uint64_t *>(from), units,
                                                                      static_cast<uint64_t *>(to), to_units, ctr);
    },
    "node rehash into %llu slots overflowed a probe sequence",
    "card-set table full: %llu nodes + %llu new vs %llu slots (max_node_bytes=%llu)"};
static const TableDesc REALISTIC_TABLE_DESC = {
    64, 1, ~0ull, 0.6, 4,
    [](const void *from, uint64_t units, void *to, uint64_t to_units, Counters *ctr, cudaStream_t st) {
        r_rehash_kernel<<<nblk((int64_t)units), TILE, 0, st>>>(static_cast<const RBucket *>(from), units,
                                                                static_cast<RBucket *>(to), to_units, ctr);
    },
    "realistic table rehash into %llu buckets overflowed a probe sequence",
    "realistic visited table full: %llu states + %llu candidates vs %llu buckets (max_table_bytes=%llu)"};
static const TableDesc RBATCH_TABLE_DESC = {
    64, 1, ~0ull, 0.6, 4,
    [](const void *from, uint64_t units, void *to, uint64_t to_units, Counters *ctr, cudaStream_t st) {
        rb_rehash_kernel<<<nblk((int64_t)units), TILE, 0, st>>>(static_cast<const RBucket *>(from), units,
                                                                 static_cast<RBucket *>(to), to_units, ctr);
    },
    "batch table rehash into %llu buckets overflowed a probe sequence",
    "batch visited table full: %llu states + %llu candidates vs %llu buckets (max_table_bytes=%llu)"};
// bucket ids are u32 with R_DEAD = 2^32 - 1 reserved: at most 2^32 - 1 buckets (128 GiB)
static const TableDesc SBATCH_TABLE_DESC = {
    32, 1, 0xFFFFFFFFull, 0.6, 4,
    [](const void *from, uint64_t units, void *to, uint64_t to_units, Counters *ctr, cudaStream_t st) {
        sb_rehash_kernel<<<nblk((int64_t)units), TILE, 0, st>>>(static_cast<const SBucket *>(from), units,
                                                                 static_cast<SBucket *>(to), to_units, ctr);
    },
    "speedrun batch table rehash into %llu buckets overflowed a probe sequence",
    "speedrun batch visited table full: %llu states + %llu candidates vs %llu buckets (max_table_bytes=%llu)"};

// A visited set on the device: an open-addressing table that grows by rehashing into one twice its size.  It counts
// its own entries, those of an insert that failed part way included, so that clear() can skip a table that holds none.
struct VisitTable {
    const TableDesc &d;
    void *p = nullptr;
    uint64_t units = 0, max_bytes = 0, occ = 0;
    explicit VisitTable(const TableDesc &desc) : d(desc) {}
    ~VisitTable() { if (p) cudaFree(p); }
    template <class T> T *as() const { return static_cast<T *>(p); }
    uint64_t slots() const { return units * d.unit_slots; }
    // a new, empty table of n units in place of the old one
    cudaError_t alloc(uint64_t n, cudaStream_t st) {
        if (p) cudaFree(p);
        p = nullptr;
        units = occ = 0;
        cudaError_t e = cudaMalloc(&p, n * d.unit_bytes);
        if (e != cudaSuccess) p = nullptr;
        else e = cudaMemsetAsync(p, 0, n * d.unit_bytes, st);
        if (e == cudaSuccess) units = n;
        return e;
    }
    cudaError_t clear(cudaStream_t st) {
        const cudaError_t e = occ ? cudaMemsetAsync(p, 0, units * d.unit_bytes, st) : cudaSuccess;
        if (e == cudaSuccess) occ = 0;
        return e;
    }
    int grow(spl_ctx *c, uint64_t need, cudaStream_t st);  // room for `need` more entries (if memory allows)
};

struct spl_ctx {
    int device = 0;
    std::string err;
    // visited sets: the key table (BFS, the reference's hash identity, externally drawn noise and the stage operators),
    // the card-set node table of the grouped level (spl_m2.cuh), the realistic level's table and the (game, key) tables
    // of the batched realistic and speedrun levels (all three allocated on first use)
    VisitTable key{KEY_TABLE_DESC}, nodes{NODE_TABLE_DESC}, rtab{REALISTIC_TABLE_DESC}, rbtab{RBATCH_TABLE_DESC},
        sbtab{SBATCH_TABLE_DESC};
    uint64_t occupied = 0;  // visited states: those of the last solve, plus what stage operators added to the key table
    uint32_t epoch = 0;
    uint64_t chunk_parents = 0;
    bool chunk_user = false;  // chunk_parents was set by the caller (spl_config), not the default
    uint64_t link_budget = 0;          // device bytes a solver may hold in parent-link columns before it spills (0: no limit)
    uint64_t spilled_bytes = 0;        // link-column bytes moved to pinned host memory so far
    uint16_t *d_gemrank = nullptr;
    uint16_t *d_rankgems = nullptr;   // inverse of d_gemrank
    DevBuf ntk8, boff2, run_start, run_wpre, cls_list;
    // constant tables
    DevTables *d_tabs = nullptr;
    uint32_t *d_takes_idx = nullptr;
    uint16_t *d_takes_edges = nullptr;
    uint32_t *d_takes_pk = nullptr;     // HostTables::takes_pk
    uint64_t *d_take_rows = nullptr;    // HostTables::take_rows
    double *d_lut = nullptr;
    ScoreLuts luts{};
    // formula heuristics (spl_add_formula): device formula table (allocated with the first formula) and one
    // power table per distinct (feature, exponent bits) pair
    FormDev *d_forms = nullptr;
    int n_forms = 0;
    std::vector<std::pair<std::pair<int, uint64_t>, double *>> pow_tabs;
    uint64_t pow_bytes = 0;
    // scalars
    Counters *d_ctr = nullptr, *h_ctr = nullptr;
    SelState *d_sel = nullptr, *h_sel = nullptr;
    uint32_t *d_hist = nullptr;
    ScoreDict *d_dict = nullptr, *d_dict2 = nullptr;  // d_dict2: the merged (global) dictionary of the sharded cut
    unsigned long long *d_dest = nullptr;             // [3][MAX_RANKS]: per-destination record counts / write cursors / base pointers
    int dict_skip = 0;
    int identity = IDENT_KEY;  // visited-table identity of the speedrun solver (spl_set_identity)  // levels left before the dictionary path is tried again after a miss
    DevBuf status[3];
    // scratch
    DevBuf off, cand_slot, tmp_rec, tmp_rec2, sk, y[2], idx[2], kl[2], kh[2], matrix, matrix2, os_hist, os_status;
    DevBuf pool_front, pool_uniq, pool_grank;  // frontier buffers lent to the active solver
    DevBuf rcfg, rcand, rvmask, ridx64, rtmp;  // realistic mode scratch
    DevBuf rkeys, rperm;       // spl_rroute_keys: packed keys of the candidates, their (owner, arrival) permutation
    int64_t rroute_n = -1;     // candidates of the last spl_rroute_keys (its permutation lives in rperm)
    spl_rconfig rcfg_host{};   // what c->rcfg holds (valid when rcfg_have)
    bool rcfg_have = false;
    uint64_t rslots_hint = 0;  // spl_config.table_slots: the first size of the realistic table, in buckets
    std::vector<DevBuf *> pool_links;  // link columns of finished solves, reused by the next one
    cudaEvent_t ev[8]{};
    long long launches = 0, h2d_bytes = 0, d2h_bytes = 0;
    int64_t dtopk_n = 0;       // distributed top-k: elements staged by spl_dtopk_begin
    int64_t route_n = -1;      // candidates of the last spl_route_keys (its permutation lives in idx[1])
    const void *active = nullptr;  // the live spl_solver: it owns the visited set, the pool buffers and the scratch
    bool rcfg_dirty = false;       // a stage operator re-uploaded the realistic config since the live solver's upload
    bool dtopk_recs = false;
    const uint64_t *dtopk_keys = nullptr;  // caller-owned [n][2] key array of the distributed top-k
};

static int fail(spl_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf; else g_create_error = buf;
    return code;
}
// stage operators that rewrite the visited set / identity must not run under a live solver
#define NO_LIVE_SOLVER(c, what)                                                                                   \
    do {                                                                                                          \
        if ((c)->active) return fail(c, SPL_E_STATE, what ": a solver is open on this context (destroy it first)"); \
    } while (0)
#define CK(c, call)                                                                             \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            cudaGetLastError();                                                                 \
            return fail(c, e_ == cudaErrorMemoryAllocation ? SPL_E_NOMEM : SPL_E_CUDA, "%s: %s (%s:%d)", #call, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                            \
        }                                                                                       \
    } while (0)
#define CKS(c, expr)              \
    do {                          \
        int s_ = (expr);          \
        if (s_ != SPL_OK) return s_; \
    } while (0)

// heuristic ids: a formula id (SPL_H_FORMULA_BASE + k) must name a formula registered on the context; every other id
// keeps its meaning (built-ins, and the fallback to simple for the rest)
static inline bool is_formula_id(int32_t h) { return h >= SPL_H_FORMULA_BASE && h < SPL_H_FORMULA_BASE + SPL_MAX_FORMULAS; }
static int check_heuristic(spl_ctx *c, const char *fn, int32_t h) {
    if (is_formula_id(h) && h - SPL_H_FORMULA_BASE >= c->n_forms)
        return fail(c, SPL_E_INVALID, "%s: heuristic %d is a formula id that is not registered on this context (%d formulas)", fn,
                    h, c->n_forms);
    return SPL_OK;
}

// every entry point: select the context's device and drop any stale non-sticky error another library left in this
// thread's runtime state (the launch checks below read cudaGetLastError, which would otherwise report it as ours)
static inline cudaError_t enter_device(spl_ctx *c) {
    const cudaError_t e = cudaSetDevice(c->device);
    if (e == cudaSuccess) cudaGetLastError();
    return e;
}
static inline int bitlen(uint64_t x) { return x ? 64 - __builtin_clzll(x) : 0; }

extern "C" {

int32_t spl_abi_version(void) { return SPL_ABI_VERSION; }

const char *spl_last_error(const spl_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

const uint32_t *spl_deck_table(int32_t *n_cards) {
    if (n_cards) *n_cards = SPL_NUM_CARDS;
    return SPL_DECK_PACKED;
}

int32_t spl_host_takes(const uint8_t gems[5], uint8_t out[100 * 5]) {
    const HostTables &T = host_tables();
    uint32_t key = 0;
    for (int c = 0; c < NCOL; ++c) {
        if (gems[c] > 7) return SPL_E_INVALID;
        key |= (uint32_t)gems[c] << (3 * c);
    }
    const uint32_t e = T.takes_idx[key], n = e & 0xff, off = e >> 8;
    for (uint32_t i = 0; i < n; ++i)
        for (int c = 0; c < NCOL; ++c) out[i * 5 + c] = (T.takes_edges[off + i] >> (3 * c)) & 7;
    return (int32_t)n;
}

int32_t spl_host_buys(const uint8_t key[5], uint8_t out[90]) {
    const HostTables &T = host_tables();
    uint64_t lo = ~0ull, hi = ~0ull;
    for (int c = 0; c < NCOL; ++c) {
        if (key[c] > 7) return SPL_E_INVALID;
        lo &= T.dev.buy_lo[c][key[c]];
        hi &= T.dev.buy_hi[c][key[c]];
    }
    int n = 0;
    for (int i = 0; i < SPL_NUM_CARDS; ++i) {
        const int b = 15 + i;
        if (b < 64 ? (lo >> b) & 1 : (hi >> (b - 64)) & 1) out[n++] = (uint8_t)i;
    }
    return n;
}

// ------------------------------------------------------------------ context
int32_t spl_create(const spl_config *cfg, spl_ctx **out) {
    if (!cfg || !out) return fail(nullptr, SPL_E_INVALID, "spl_create: null argument");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(nullptr, SPL_E_NODEVICE, "spl_create: no CUDA device (%s); this library has no CPU fallback",
                    cudaGetErrorString(e));
    }
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, SPL_E_INVALID, "spl_create: bad device %d", cfg->device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess || prop.major != 10)
        return fail(nullptr, SPL_E_NODEVICE, "spl_create: device %d is sm_%d%d; this build is sm_100a only", cfg->device,
                    prop.major, prop.minor);
    spl_ctx *c = new spl_ctx();
    c->device = cfg->device;
#define CKC(call)                                                                                             \
    do {                                                                                                      \
        cudaError_t e2_ = (call);                                                                             \
        if (e2_ != cudaSuccess) {                                                                             \
            cudaGetLastError();                                                                               \
            int r_ = fail(nullptr, e2_ == cudaErrorMemoryAllocation ? SPL_E_NOMEM : SPL_E_CUDA, "%s: %s", #call, \
                          cudaGetErrorString(e2_));                                                           \
            delete c;                                                                                         \
            return r_;                                                                                        \
        }                                                                                                     \
    } while (0)
    CKC(cudaSetDevice(c->device));
    size_t free_b = 0, total_b = 0;
    CKC(cudaMemGetInfo(&free_b, &total_b));
    c->key.max_bytes = c->rtab.max_bytes = c->rbtab.max_bytes = c->sbtab.max_bytes = cfg->max_table_bytes ? cfg->max_table_bytes : (uint64_t)(free_b * 0.6);
    c->chunk_user = cfg->chunk_parents != 0;
    c->chunk_parents = cfg->chunk_parents ? std::min<uint64_t>(cfg->chunk_parents, MAX_CHUNK_PARENTS) : (4ull << 20);
    c->chunk_parents = std::max<uint64_t>(c->chunk_parents, TILE);
    const HostTables &T = host_tables();
    CKC(cudaMalloc(&c->d_tabs, sizeof(DevTables)));
    CKC(cudaMemcpy(c->d_tabs, &T.dev, sizeof(DevTables), cudaMemcpyHostToDevice));
    CKC(cudaMalloc(&c->d_takes_idx, T.takes_idx.size() * 4));
    CKC(cudaMemcpy(c->d_takes_idx, T.takes_idx.data(), T.takes_idx.size() * 4, cudaMemcpyHostToDevice));
    CKC(cudaMalloc(&c->d_takes_edges, T.takes_edges.size() * 2));
    CKC(cudaMemcpy(c->d_takes_edges, T.takes_edges.data(), T.takes_edges.size() * 2, cudaMemcpyHostToDevice));
    CKC(cudaMalloc(&c->d_takes_pk, T.takes_pk.size() * 4));
    CKC(cudaMemcpy(c->d_takes_pk, T.takes_pk.data(), T.takes_pk.size() * 4, cudaMemcpyHostToDevice));
    CKC(cudaMalloc(&c->d_take_rows, T.take_rows.size() * 8));
    CKC(cudaMemcpy(c->d_take_rows, T.take_rows.data(), T.take_rows.size() * 8, cudaMemcpyHostToDevice));
    const size_t n_lut = T.lut_pts.size() + T.lut_saved.size() + T.lut_small.size();
    CKC(cudaMalloc(&c->d_lut, n_lut * 8));
    CKC(cudaMemcpy(c->d_lut, T.lut_pts.data(), T.lut_pts.size() * 8, cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_lut + T.lut_pts.size(), T.lut_saved.data(), T.lut_saved.size() * 8, cudaMemcpyHostToDevice));
    CKC(cudaMemcpy(c->d_lut + T.lut_pts.size() + T.lut_saved.size(), T.lut_small.data(), T.lut_small.size() * 8,
                   cudaMemcpyHostToDevice));
    c->luts.pts = c->d_lut;
    c->luts.saved = c->d_lut + T.lut_pts.size();
    c->luts.small = c->d_lut + T.lut_pts.size() + T.lut_saved.size();
    CKC(cudaMalloc(&c->d_gemrank, T.gemrank.size() * 2));
    CKC(cudaMemcpy(c->d_gemrank, T.gemrank.data(), T.gemrank.size() * 2, cudaMemcpyHostToDevice));
    {
        std::vector<uint16_t> inv(GEM_STATES, 0);
        for (size_t g = 0; g < T.gemrank.size(); ++g)
            if (T.gemrank[g] != 0xFFFF) inv[T.gemrank[g]] = (uint16_t)g;
        CKC(cudaMalloc(&c->d_rankgems, inv.size() * 2));
        CKC(cudaMemcpy(c->d_rankgems, inv.data(), inv.size() * 2, cudaMemcpyHostToDevice));
    }
    CKC(cudaMalloc(&c->d_ctr, sizeof(Counters)));
    CKC(cudaMallocHost(&c->h_ctr, sizeof(Counters)));
    CKC(cudaMalloc(&c->d_sel, sizeof(SelState)));
    CKC(cudaMallocHost(&c->h_sel, sizeof(SelState)));
    CKC(cudaMalloc(&c->d_hist, SEL_BINS * 4));
    CKC(cudaMemset(c->d_hist, 0, SEL_BINS * 4));
    CKC(cudaMalloc(&c->d_dict, sizeof(ScoreDict)));
    for (auto &ev : c->ev) CKC(cudaEventCreate(&ev));
    CKC(cudaFuncSetAttribute(expand_kernel<MODE_PROBE, IDENT_KEY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ExpandSmem2)));
    CKC(cudaFuncSetAttribute(expand_kernel<MODE_PROBE, IDENT_PYHASH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ExpandSmem2)));
    CKC(cudaFuncSetAttribute(expand_kernel<MODE_LIST, IDENT_KEY>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(ExpandSmem2)));
    CKC(cudaFuncSetAttribute(m2_buys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BuySmem)));
    CKC(cudaFuncSetAttribute(m2_group_warp_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)offsetof(WarpSmem, bsort)));
    CKC(cudaFuncSetAttribute(m2_group_warp_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(WarpSmem)));
    CKC(cudaFuncSetAttribute(m2_group_big_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BigSmem)));
    CKC(cudaFuncSetAttribute(m2_group_big_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BigSmem)));
    CKC(cudaFuncSetAttribute(os_scatter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)offsetof(OsSmem, stage_p)));
    CKC(cudaFuncSetAttribute(os_scatter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(OsSmem)));
    CKC(cudaFuncSetAttribute(gs_buys_route_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(RouteSmem)));
    CKC(cudaMalloc(&c->d_dict2, sizeof(ScoreDict)));
    CKC(cudaMalloc(&c->d_dest, 3 * MAX_RANKS * 8));
    {
        c->nodes.max_bytes = cfg->max_node_bytes ? cfg->max_node_bytes : (uint64_t)(free_b * 0.5);
        uint64_t nn = cfg->node_slots ? cfg->node_slots : (1ull << 12);
        nn = std::max<uint64_t>(std::min<uint64_t>(nn, c->nodes.max_bytes / (NODE_WORDS * 8)), 64);
        CKC(c->nodes.alloc(nn, 0));
    }
    c->rslots_hint = cfg->table_slots;
    uint64_t slots = cfg->table_slots ? cfg->table_slots : (1ull << 22);
    slots = std::min<uint64_t>(slots, c->key.max_bytes / 64 * BUCKET_SLOTS);
    slots = std::max<uint64_t>(slots, 1024);
    CKC(c->key.alloc(buckets_for(slots), 0));
    CKC(cudaDeviceSynchronize());
#undef CKC
    *out = c;
    return SPL_OK;
}

int32_t spl_destroy(spl_ctx *c) {
    if (!c) return SPL_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    cudaFree(c->d_tabs); cudaFree(c->d_takes_idx); cudaFree(c->d_takes_edges); cudaFree(c->d_takes_pk); cudaFree(c->d_take_rows);
    cudaFree(c->d_lut); cudaFree(c->d_ctr); cudaFreeHost(c->h_ctr); cudaFree(c->d_sel); cudaFreeHost(c->h_sel);
    cudaFree(c->d_hist); cudaFree(c->d_dict); cudaFree(c->d_dict2); cudaFree(c->d_dest); cudaFree(c->d_gemrank); cudaFree(c->d_rankgems);
    cudaFree(c->d_forms);
    for (auto &t : c->pow_tabs) cudaFree(t.second);
    for (auto *b : c->pool_links) delete b;
    for (auto &ev : c->ev) if (ev) cudaEventDestroy(ev);
    delete c;
    return SPL_OK;
}

static int reset_visited(spl_ctx *c, cudaStream_t st) {
    CK(c, enter_device(c));
    CK(c, c->key.clear(st));
    CK(c, c->nodes.clear(st));
    c->occupied = 0;
    c->epoch = 0;
    return SPL_OK;
}

int32_t spl_reset_visited(spl_ctx *c, void *stream) {
    if (!c) return SPL_E_INVALID;
    NO_LIVE_SOLVER(c, "spl_reset_visited");
    return reset_visited(c, (cudaStream_t)stream);
}

int32_t spl_set_identity(spl_ctx *c, int32_t identity) {
    if (!c) return SPL_E_INVALID;
    if (identity != SPL_IDENT_KEY && identity != SPL_IDENT_PYHASH) return fail(c, SPL_E_INVALID, "spl_set_identity: unknown identity %d", identity);
    NO_LIVE_SOLVER(c, "spl_set_identity");
    c->identity = identity == SPL_IDENT_PYHASH ? IDENT_PYHASH : IDENT_KEY;
    return SPL_OK;
}

int32_t spl_set_link_budget(spl_ctx *c, uint64_t device_bytes) {
    if (!c) return SPL_E_INVALID;
    NO_LIVE_SOLVER(c, "spl_set_link_budget");
    c->link_budget = device_bytes;
    return SPL_OK;
}

int32_t spl_spilled_bytes(spl_ctx *c, int64_t *n_host) {
    if (!c || !n_host) return SPL_E_INVALID;
    *n_host = (int64_t)c->spilled_bytes;
    return SPL_OK;
}

int32_t spl_pyhash(spl_ctx *c, const spl_key *keys, int64_t n, uint64_t *out, void *stream) {
    if (!c || n < 0 || (n && (!keys || !out))) return fail(c, SPL_E_INVALID, "spl_pyhash: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    pyhash_kernel<<<nblk(n), TILE, 0, st>>>(keys, n, out);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_visited_count(spl_ctx *c, int64_t *n_host) {
    if (!c || !n_host) return SPL_E_INVALID;
    *n_host = (int64_t)c->occupied;
    return SPL_OK;
}

int32_t spl_launch_count(spl_ctx *c, int64_t *n_host) {
    if (!c || !n_host) return SPL_E_INVALID;
    *n_host = c->launches;
    return SPL_OK;
}

int32_t spl_transfer_bytes(spl_ctx *c, int64_t *h2d_host, int64_t *d2h_host) {
    if (!c || !h2d_host || !d2h_host) return SPL_E_INVALID;
    *h2d_host = c->h2d_bytes;
    *d2h_host = c->d2h_bytes;
    return SPL_OK;
}

// ------------------------------------------------------------------ internal helpers
static int zero_ctr(spl_ctx *c, cudaStream_t st) {
    Counters z;
    memset(&z, 0, sizeof z);
    z.sk_min = ~0ull;
    z.goal_rank = 0x7fffffffffffffffll;
    z.key_and[0] = z.key_and[1] = ~0ull;
    *c->h_ctr = z;
    CK(c, cudaMemcpyAsync(c->d_ctr, c->h_ctr, sizeof z, cudaMemcpyHostToDevice, st));
    c->h2d_bytes += sizeof z;
    return SPL_OK;
}
static int read_ctr(spl_ctx *c, cudaStream_t st) {
    CK(c, cudaMemcpyAsync(c->h_ctr, c->d_ctr, sizeof(Counters), cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    c->d2h_bytes += sizeof(Counters);
    return SPL_OK;
}
static int reset_ticket(spl_ctx *c, int id, cudaStream_t st) {
    CK(c, cudaMemsetAsync(&c->d_ctr->ticket[id], 0, 4, st));
    return SPL_OK;
}
static int prep_status(spl_ctx *c, int which, size_t ntiles, cudaStream_t st) {
    CK(c, c->status[which].ensure((ntiles + 1) * 8, 0, st));
    CK(c, cudaMemsetAsync(c->status[which].p, 0, (ntiles + 1) * 8, st));
    return SPL_OK;
}

// grow so that `need` more entries keep the load factor (if memory allows)
int VisitTable::grow(spl_ctx *c, uint64_t need, cudaStream_t st) {
    while ((double)(occ + need) > d.load * (double)slots()) {
        uint64_t nu = std::min<uint64_t>(units * 2, d.max_units);
        if (nu * d.unit_bytes > max_bytes) nu = max_bytes / d.unit_bytes;
        if (nu <= units + units / 8) break;  // cannot grow meaningfully
        void *nt = nullptr;
        cudaError_t e = cudaMalloc(&nt, nu * d.unit_bytes);
        if (e != cudaSuccess) { cudaGetLastError(); break; }
        CK(c, cudaMemsetAsync(nt, 0, nu * d.unit_bytes, st));
        d.rehash(p, units, nt, nu, c->d_ctr, st);
        ++c->launches;
        CK(c, cudaGetLastError());
        unsigned int rehash_err = 0;  // read the flag now: callers zero the counters before their own launches
        CK(c, cudaMemcpyAsync(&rehash_err, &c->d_ctr->error, 4, cudaMemcpyDeviceToHost, st));
        CK(c, cudaStreamSynchronize(st));
        if (rehash_err) {
            cudaFree(nt);
            return fail(c, SPL_E_TABLE_FULL, d.rehash_msg, (unsigned long long)nu);
        }
        cudaFree(p);
        p = nt;
        units = nu;
    }
    if (occ + need / d.full_div > slots() - slots() / 16)
        return fail(c, SPL_E_TABLE_FULL, d.full_msg, (unsigned long long)occ, (unsigned long long)need,
                    (unsigned long long)slots(), (unsigned long long)max_bytes);
    return SPL_OK;
}

static int next_epoch(spl_ctx *c, uint64_t &tag) {
    if (c->epoch >= TAG_MAX) return fail(c, SPL_E_STATE, "epoch tag exhausted");
    tag = ++c->epoch;
    return SPL_OK;
}

// count + offsets for parents front[0..n): leaves total in h_ctr->total_cands (synchronises)
static int run_count(spl_ctx *c, const Rec *front, int64_t n, cudaStream_t st) {
    const unsigned nt = nblk(n);
    CK(c, c->off.ensure((size_t)n * 4 + 4, 0, st));
    CKS(c, prep_status(c, 0, nt, st));
    CKS(c, reset_ticket(c, 0, st));
    count_scan_kernel<<<nt, TILE, 0, st>>>(front, n, c->d_tabs, c->d_takes_idx, c->off.as<uint32_t>(),
                                            c->status[0].as<uint64_t>(), c->d_ctr, 0);
    ++c->launches;
    CK(c, cudaGetLastError());
    return read_ctr(c, st);
}

// How the beam cut orders the states that tie on score.
enum CutTies {
    TIES_ARRIVAL,      // arrival order, the input being in arrival order (stable policy)
    TIES_KEY,          // larger key first (det policy)
    TIES_KEY_ORDERED,  // larger key first, the input being in key order already: only the score is sorted
    TIES_LINK,         // arrival order read from the records' link words, the input being unordered (grouped level)
};
struct CutMode {
    CutTies ties = TIES_ARRIVAL;
    int link_bits = 0;  // TIES_LINK: the tie word is 2^link_bits - 1 - link
    bool by_key() const { return ties != TIES_ARRIVAL; }                      // a key threshold splits the ties
    bool sorts_keys() const { return ties == TIES_KEY || ties == TIES_LINK; }  // the rank sort has key passes
    int lt() const { return ties == TIES_LINK ? link_bits : 0; }
};

// key policies: split the score ties at the threshold (d_sel->prefix) by key, larger first
static int select_ties_by_key(spl_ctx *c, const uint64_t *sk, const uint64_t *kb, int ks, int64_t n, int64_t k,
                              uint64_t sk_min, CutMode mode, cudaStream_t st) {
    const unsigned grid = std::min<unsigned>(nblk(n), 148 * 8);
    const int lt = mode.lt();
    if (lt) {
        // arrival-order ties: collect the tie words (2^lt - 1 - link) of the threshold score once, then select among them
        const int64_t ntie = (int64_t)c->h_sel->tie_count;
        CK(c, c->rtmp.ensure((size_t)ntie * 8 + 8, 0, st));
        CK(c, cudaMemsetAsync(&c->d_ctr->n_ties, 0, 8, st));
        tie_collect_kernel<<<grid, TILE, 0, st>>>(sk, kb, ks, n, sk_min, c->d_sel, lt, c->rtmp.as<uint64_t>(), c->d_ctr);
        ++c->launches;
        const unsigned tgrid = std::min<unsigned>(nblk(ntie), 148 * 8);
        int top = lt, first = 1;
        while (top > 0) {
            const int bits = std::min(SEL_BITS, top), shift = top - bits;
            sel_hist_kernel<3><<<tgrid, TILE, 0, st>>>(nullptr, c->rtmp.as<uint64_t>(), 1, ntie, 0, shift, bits, first, c->d_sel, c->d_hist);
            sel_pick_kernel<<<1, 1024, 0, st>>>(c->d_hist, 2, shift, first, 0, (uint64_t)k, c->d_sel);
            c->launches += 2;
            first = 0;
            top = shift;
        }
    } else
    for (int word = 1; word <= 2; ++word) {
        int top = word == 1 ? 41 : 64, first = 1;
        while (top > 0) {
            const int bits = std::min(SEL_BITS, top), shift = top - bits;
            if (word == 1) sel_hist_kernel<1><<<grid, TILE, 0, st>>>(sk, kb, ks, n, sk_min, shift, bits, first, c->d_sel, c->d_hist);
            else sel_hist_kernel<2><<<grid, TILE, 0, st>>>(sk, kb, ks, n, sk_min, shift, bits, first, c->d_sel, c->d_hist);
            sel_pick_kernel<<<1, 1024, 0, st>>>(c->d_hist, word, shift, first, 0, (uint64_t)k, c->d_sel);
            c->launches += 2;
            first = 0;
            top = shift;
        }
    }
    CK(c, cudaGetLastError());
    c->h_sel->tie_count = ~0ull;  // marks "threshold key valid"
    return SPL_OK;
}

// radix select of the k-th largest element under (score desc[, key desc]); leaves the thresholds and
// the tie quota in d_sel / h_sel (score in x = sk - sk_min space).
static int run_select(spl_ctx *c, const uint64_t *sk, const uint64_t *kb, int ks, int64_t n, int64_t k, uint64_t sk_min,
                      uint64_t sk_max, CutMode mode, cudaStream_t st) {
    const int nbits = bitlen(sk_max - sk_min);
    const unsigned grid = std::min<unsigned>(nblk(n), 148 * 8);
    memset(c->h_sel, 0, sizeof(SelState));
    c->h_sel->k_rem = (unsigned long long)k;
    c->h_sel->tie_count = (unsigned long long)n;  // nbits == 0: every score equal
    c->h_sel->rank_t = ~0ull;
    CK(c, cudaMemcpyAsync(c->d_sel, c->h_sel, sizeof(SelState), cudaMemcpyHostToDevice, st));
    int top = nbits, first = 1, init_k = 1;
    while (top > 0) {
        const int bits = std::min(SEL_BITS, top), shift = top - bits;
        sel_hist_kernel<0><<<grid, TILE, 0, st>>>(sk, kb, ks, n, sk_min, shift, bits, first, c->d_sel, c->d_hist);
        sel_pick_kernel<<<1, 1024, 0, st>>>(c->d_hist, 0, shift, first, init_k, (uint64_t)k, c->d_sel);
        c->launches += 2;
        first = init_k = 0;
        top = shift;
    }
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(c->h_sel, c->d_sel, sizeof(SelState), cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    c->d2h_bytes += sizeof(SelState);
    if (mode.by_key() && c->h_sel->k_rem < c->h_sel->tie_count) CKS(c, select_ties_by_key(c, sk, kb, ks, n, k, sk_min, mode, st));
    return SPL_OK;
}

// Dictionary select (few distinct scores): count the distinct scores, rank them, find the k-th largest
// element.  Leaves d_sel / h_sel as run_select does plus rank_t; *used = 0 when the level has more
// than DICT_MAX distinct scores (nothing decided: the caller falls back to the radix select).
static int run_dict_select(spl_ctx *c, const uint64_t *sk, const uint64_t *kb, int ks, int64_t n, int64_t k,
                           uint64_t sk_min, CutMode mode, int *used, cudaStream_t st, int keep_all = -1) {
    if (keep_all < 0) keep_all = k >= n;
    *used = 0;
    if (c->dict_skip > 0) { --c->dict_skip; return SPL_OK; }
    const unsigned grid = std::min<unsigned>(nblk(n), 148 * 8);
    CK(c, cudaMemsetAsync(c->d_dict->key, 0xFF, sizeof(c->d_dict->key), st));
    CK(c, cudaMemsetAsync(c->d_dict->cnt, 0, sizeof(ScoreDict) - sizeof(c->d_dict->key), st));
    memset(c->h_sel, 0, sizeof(SelState));
    c->h_sel->rank_t = ~0ull;
    CK(c, cudaMemcpyAsync(c->d_sel, c->h_sel, sizeof(SelState), cudaMemcpyHostToDevice, st));
    dict_build_kernel<<<grid, TILE, 0, st>>>(sk, n, c->d_dict);
    dict_rank_kernel<<<1, 1024, 0, st>>>(c->d_dict, (uint64_t)k, sk_min, c->d_sel);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(c->h_sel, c->d_sel, sizeof(SelState), cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    c->d2h_bytes += sizeof(SelState);
    if (c->h_sel->rank_t == ~0ull) {
        c->dict_skip = 3;
        return SPL_OK;
    }
    *used = 1;
    if (mode.by_key() && !keep_all && c->h_sel->k_rem < c->h_sel->tie_count) CKS(c, select_ties_by_key(c, sk, kb, ks, n, k, sk_min, mode, st));
    return SPL_OK;
}

static int onesweep_sort(spl_ctx *c, uint64_t *const k[2], uint32_t *const pl[2], int64_t n, int lo_bit, int nbits, int *cur, cudaStream_t st);

// one stable LSD pass over `kept` elements: digit = (dig >> shift) & 255
static int sort_pass(spl_ctx *c, int wide, int cur, const uint64_t *dig, int64_t kept, int shift, unsigned nt,
                     size_t msz, cudaStream_t st) {
    const unsigned st_tiles = nblk((int64_t)msz, TILE * SCAN_ITEMS);
    sort_hist_kernel<<<nt, TILE, 0, st>>>(dig, kept, shift, c->matrix.as<uint32_t>(), nt);
    CKS(c, prep_status(c, 1, st_tiles, st));
    CKS(c, reset_ticket(c, 2, st));
    scan_u32_kernel<<<st_tiles, TILE, 0, st>>>(c->matrix.as<uint32_t>(), c->matrix2.as<uint32_t>(), (int64_t)msz,
                                                c->status[1].as<uint64_t>(), c->d_ctr, 2);
    if (wide)
        sort_scatter_kernel<true><<<nt, TILE, 0, st>>>(dig, c->y[cur].as<uint64_t>(), c->idx[cur].as<uint32_t>(), kept, shift,
                                                        c->matrix2.as<uint32_t>(), nt, c->y[cur ^ 1].as<uint64_t>(),
                                                        c->idx[cur ^ 1].as<uint32_t>(), c->kl[cur].as<uint64_t>(),
                                                        c->kh[cur].as<uint64_t>(), c->kl[cur ^ 1].as<uint64_t>(),
                                                        c->kh[cur ^ 1].as<uint64_t>());
    else
        sort_scatter_kernel<false><<<nt, TILE, 0, st>>>(dig, c->y[cur].as<uint64_t>(), c->idx[cur].as<uint32_t>(), kept, shift,
                                                         c->matrix2.as<uint32_t>(), nt, c->y[cur ^ 1].as<uint64_t>(),
                                                         c->idx[cur ^ 1].as<uint32_t>(), nullptr, nullptr, nullptr, nullptr);
    c->launches += 3;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

// Stable sort of the (sort word, slot) pairs c->y[*cur] / c->idx[*cur] [0, n) by the words' low `nbits` bits: one-sweep
// passes below OS_MAX_ITEMS pairs, 8-bit LSD passes at and above it.
static int sort_pairs(spl_ctx *c, int64_t n, int nbits, int *cur, cudaStream_t st) {
    if (n <= 1 || nbits <= 0) return SPL_OK;
    if (n < OS_MAX_ITEMS) {
        uint64_t *const yk[2] = {c->y[0].as<uint64_t>(), c->y[1].as<uint64_t>()};
        uint32_t *const yi[2] = {c->idx[0].as<uint32_t>(), c->idx[1].as<uint32_t>()};
        return onesweep_sort(c, yk, yi, n, 0, nbits, cur, st);
    }
    const unsigned nt = nblk(n, SORT_TILE);
    const size_t msz = (size_t)SORT_BINS * nt;
    CK(c, c->matrix.ensure(msz * 4, 0, st));
    CK(c, c->matrix2.ensure(msz * 4, 0, st));
    for (int shift = 0; shift < nbits; shift += SORT_BITS) {
        CKS(c, sort_pass(c, 0, *cur, c->y[*cur].as<uint64_t>(), n, shift, nt, msz, st));
        *cur ^= 1;
    }
    return SPL_OK;
}

// Packed beam cut by the thresholds in d_sel: one sort word per survivor (its score's rank in `dict` << link_bits | link
// word), then the (word, slot) pairs sorted ascending -- best first -- into c->y[*cur] / c->idx[*cur].  At most `cap`
// survivors.
static int cut_packed(spl_ctx *c, const uint64_t *sk, const uint64_t *kb, int ks, int64_t n, int64_t cap, uint64_t sk_min,
                      int keep_all, int all_ties, const ScoreDict *dict, int link_bits, int *cur, int64_t *kept_out,
                      cudaStream_t st) {
    for (int b = 0; b < 2; ++b) {
        CK(c, c->y[b].ensure((size_t)cap * 8 + 8, 0, st));
        CK(c, c->idx[b].ensure((size_t)cap * 4 + 4, 0, st));
    }
    const unsigned ct = nblk(n, TILE * CUTP_ITEMS);
    CKS(c, prep_status(c, 2, ct, st));
    CKS(c, zero_ctr(c, st));
    cut_pack_kernel<<<ct, TILE, 0, st>>>(sk, kb, ks, n, sk_min, keep_all, all_ties, c->d_sel, dict, link_bits, c->y[0].as<uint64_t>(),
                                          c->idx[0].as<uint32_t>(), c->status[2].as<uint64_t>(), c->d_ctr, 1);
    ++c->launches;
    CK(c, cudaGetLastError());
    uint64_t last = 0;  // survivors written: the inclusive prefix published by the last cut tile
    CK(c, cudaMemcpyAsync(&last, c->status[2].as<uint64_t>() + (ct - 1), 8, cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    c->d2h_bytes += 8;
    const int64_t kept = (int64_t)(last & ((1ull << 62) - 1));
    if (kept > cap) return fail(c, SPL_E_CUDA, "internal: cut kept %lld > capacity %lld", (long long)kept, (long long)cap);
    *cur = 0;
    *kept_out = kept;
    return sort_pairs(c, kept, bitlen(c->h_sel->rank_t) + link_bits, cur, st);
}

// beam cut + rank sort by the thresholds currently in d_sel / h_sel (x-space score threshold `prefix`, arrival quota
// `k_rem` for arrival ties, key threshold khi/klo for key ties).  Arrival ties: arrival-order cut, stable descending sort
// by score.  Key ties: cut and sort by (score desc, key desc).  On return idx[*which] holds the kept source indices in
// rank order.
static int do_cut_sort(spl_ctx *c, const uint64_t *sk, const uint64_t *kb, int ks, int64_t n, int64_t cap_kept, int keep_all,
                       int all_ties, uint64_t sk_min, uint64_t sk_max, CutMode mode, int use_dict, int *which, int64_t *kept_out,
                       cudaStream_t st) {
    if (mode.ties == TIES_LINK && use_dict)
        return cut_packed(c, sk, kb, ks, n, cap_kept, sk_min, keep_all, all_ties, c->d_dict, mode.link_bits, which, kept_out, st);
    int64_t kept = cap_kept;
    const uint64_t T = keep_all ? 0 : c->h_sel->prefix;
    for (int b = 0; b < 2; ++b) {
        CK(c, c->y[b].ensure((size_t)kept * 8 + 8, 0, st));
        CK(c, c->idx[b].ensure((size_t)kept * 4 + 4, 0, st));
        if (mode.by_key()) {
            CK(c, c->kl[b].ensure((size_t)kept * 8 + 8, 0, st));
            CK(c, c->kh[b].ensure((size_t)kept * 8 + 8, 0, st));
        }
    }
    const unsigned ct = nblk(n, TILE * CUT_ITEMS);
    CKS(c, prep_status(c, 1, ct, st));
    CKS(c, prep_status(c, 2, ct, st));
    CKS(c, reset_ticket(c, 1, st));
    uint64_t vary_lo = 0, vary_hi = 0;
    if (mode.by_key()) {
        CKS(c, zero_ctr(c, st));
        if (use_dict)
            cut_det_kernel<true><<<ct, TILE, 0, st>>>(sk, kb, ks, n, sk_min, sk_max, keep_all, all_ties, c->d_sel, c->d_dict,
                                                       c->y[0].as<uint64_t>(), c->kl[0].as<uint64_t>(), c->kh[0].as<uint64_t>(),
                                                       c->idx[0].as<uint32_t>(), c->status[2].as<uint64_t>(), c->d_ctr, 1, mode.lt(), 0);
        else
            cut_det_kernel<false><<<ct, TILE, 0, st>>>(sk, kb, ks, n, sk_min, sk_max, keep_all, all_ties, c->d_sel, nullptr,
                                                        c->y[0].as<uint64_t>(), c->kl[0].as<uint64_t>(), c->kh[0].as<uint64_t>(),
                                                        c->idx[0].as<uint32_t>(), c->status[2].as<uint64_t>(), c->d_ctr, 1, mode.lt(), 0);
        ++c->launches;
        CK(c, cudaGetLastError());
        if (mode.sorts_keys()) {  // which key bits vary among the survivors (constant digits need no sort pass)
            CKS(c, read_ctr(c, st));
            vary_lo = c->h_ctr->key_or[0] ^ c->h_ctr->key_and[0];
            vary_hi = (c->h_ctr->key_or[1] ^ c->h_ctr->key_and[1]) & HI_KEY_MASK;
        }
    } else {
        if (use_dict)
            cut_kernel<true><<<ct, TILE, 0, st>>>(sk, n, sk_min, sk_max, keep_all, c->d_sel, c->d_dict, c->y[0].as<uint64_t>(),
                                                   c->idx[0].as<uint32_t>(), c->status[1].as<uint64_t>(),
                                                   c->status[2].as<uint64_t>(), c->d_ctr, 1);
        else
            cut_kernel<false><<<ct, TILE, 0, st>>>(sk, n, sk_min, sk_max, keep_all, c->d_sel, nullptr, c->y[0].as<uint64_t>(),
                                                    c->idx[0].as<uint32_t>(), c->status[1].as<uint64_t>(),
                                                    c->status[2].as<uint64_t>(), c->d_ctr, 1);
        ++c->launches;
        CK(c, cudaGetLastError());
    }
    {   // survivors actually written, from the inclusive prefixes published by the last cut tile
        const bool quota = mode.ties == TIES_ARRIVAL && !keep_all;  // the threshold score's ties fill the arrival quota
        uint64_t last = 0, last_tie = 0;
        CK(c, cudaMemcpyAsync(&last, c->status[2].as<uint64_t>() + (ct - 1), 8, cudaMemcpyDeviceToHost, st));
        if (quota) CK(c, cudaMemcpyAsync(&last_tie, c->status[1].as<uint64_t>() + (ct - 1), 8, cudaMemcpyDeviceToHost, st));
        CK(c, cudaStreamSynchronize(st));
        c->d2h_bytes += quota ? 16 : 8;
        constexpr uint64_t VAL = (1ull << 62) - 1;
        kept = (int64_t)(last & VAL);  // key ties: kept states; arrival ties: states above the threshold
        if (quota) kept += (int64_t)std::min<uint64_t>(last_tie & VAL, c->h_sel->k_rem);
        if (kept > cap_kept) return fail(c, SPL_E_CUDA, "internal: cut kept %lld > capacity %lld", (long long)kept, (long long)cap_kept);
    }
    // y = sk_max - sk in [0, sk_max - sk_min - T], or (dictionary) the score's descending rank in [0, rank_t]
    const int nbits = use_dict ? bitlen(c->h_sel->rank_t) : bitlen((sk_max - sk_min) - T);
    int cur = 0;
    if (kept > 1 && (nbits > 0 || vary_lo || vary_hi)) {
        if (mode.sorts_keys()) {  // least significant first: key.lo, key.hi, then the score
            const unsigned nt = nblk(kept, SORT_TILE);
            const size_t msz = (size_t)SORT_BINS * nt;
            CK(c, c->matrix.ensure(msz * 4, 0, st));
            CK(c, c->matrix2.ensure(msz * 4, 0, st));
            for (int shift = 0; shift < 64; shift += SORT_BITS)
                if ((vary_lo >> shift) & 0xff) { CKS(c, sort_pass(c, 1, cur, c->kl[cur].as<uint64_t>(), kept, shift, nt, msz, st)); cur ^= 1; }
            for (int shift = 0; shift < 41; shift += SORT_BITS)
                if ((vary_hi >> shift) & 0xff) { CKS(c, sort_pass(c, 1, cur, c->kh[cur].as<uint64_t>(), kept, shift, nt, msz, st)); cur ^= 1; }
            for (int shift = 0; shift < nbits; shift += SORT_BITS) {
                CKS(c, sort_pass(c, 1, cur, c->y[cur].as<uint64_t>(), kept, shift, nt, msz, st));
                cur ^= 1;
            }
        } else {
            CKS(c, sort_pairs(c, kept, nbits, &cur, st));
        }
    }
    if (mode.ties == TIES_KEY_ORDERED && kept > 0) {  // keys were in rank order already: the stable score sort kept them so; rebuild the key words
        key_words_kernel<<<nblk(kept), TILE, 0, st>>>(c->idx[cur].as<uint32_t>(), kept, kb, ks, c->kl[cur].as<uint64_t>(),
                                                       c->kh[cur].as<uint64_t>());
        ++c->launches;
        CK(c, cudaGetLastError());
    }
    *which = cur;
    *kept_out = kept;
    return SPL_OK;
}

// n = elements of sk / recs; n_valid of them are states (the rest are unused slots, sk == 0)
static int run_cut_sort(spl_ctx *c, const uint64_t *sk, const Rec *recs, int64_t n, int64_t k, uint64_t sk_min,
                        uint64_t sk_max, CutMode mode, int *which, int64_t *kept_out, cudaStream_t st, int64_t n_valid = -1) {
    if (n_valid < 0) n_valid = n;
    const int keep_all = n_valid <= k;
    const uint64_t *kb = reinterpret_cast<const uint64_t *>(recs);
    const int ks = 4;
    int use_dict = 0;
    CKS(c, run_dict_select(c, sk, kb, ks, n, std::min(n_valid, k), sk_min, mode, &use_dict, st, keep_all));
    if (!keep_all && !use_dict) CKS(c, run_select(c, sk, kb, ks, n, k, sk_min, sk_max, mode, st));
    const int all_ties = keep_all || c->h_sel->tie_count != ~0ull;
    CKS(c, do_cut_sort(c, sk, kb, ks, n, std::min(n_valid, k), keep_all, all_ties, sk_min, sk_max, mode, use_dict, which, kept_out, st));
    if (*kept_out != std::min(n_valid, k))
        return fail(c, SPL_E_CUDA, "internal: cut kept %lld states, expected %lld", (long long)*kept_out, (long long)std::min(n_valid, k));
    return SPL_OK;
}

// ------------------------------------------------------------------ stage operators
int32_t spl_expand(spl_ctx *c, const spl_key *keys, const uint64_t *aux, int64_t n, spl_key *ck, uint64_t *ca,
                   uint64_t *cl, int64_t cap, int64_t *n_out, void *stream) {
    if (!c || !n_out || n < 0 || n > (16ll << 20)) return fail(c, SPL_E_INVALID, "spl_expand: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0) return SPL_OK;
    CK(c, c->tmp_rec.ensure((size_t)n * 32, 0, st));
    pack_rec_kernel<<<nblk(n), TILE, 0, st>>>(keys, aux, n, c->tmp_rec.as<Rec>());
    ++c->launches;
    CKS(c, zero_ctr(c, st));
    CKS(c, run_count(c, c->tmp_rec.as<Rec>(), n, st));
    const int64_t total = (int64_t)c->h_ctr->total_cands;
    *n_out = total;
    if (total > cap) return fail(c, SPL_E_CAPACITY, "spl_expand: %lld successors, capacity %lld", (long long)total, (long long)cap);
    if (total == 0) return SPL_OK;
    CK(c, c->tmp_rec2.ensure((size_t)total * 32, 0, st));
    expand_kernel<MODE_LIST, IDENT_KEY><<<nblk(n), TILE, sizeof(ExpandSmem2), st>>>(
        c->tmp_rec.as<Rec>(), n, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(), (uint32_t)total,
        nullptr, 0, 0, nullptr, c->tmp_rec2.as<Rec>(), 0, c->d_ctr);
    unpack_rec_kernel<<<nblk(total), TILE, 0, st>>>(c->tmp_rec2.as<Rec>(), total, ck, ca, cl);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaStreamSynchronize(st));
    return SPL_OK;
}

int32_t spl_dedup(spl_ctx *c, const spl_key *ck, const uint64_t *ca, int64_t n, spl_key *uk, uint64_t *ua, int64_t *usrc,
                  int64_t *n_out, void *stream) {
    if (!c || !n_out || n < 0 || n >= (1ll << 32)) return fail(c, SPL_E_INVALID, "spl_dedup: bad arguments");
    NO_LIVE_SOLVER(c, "spl_dedup");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0) return SPL_OK;
    CKS(c, zero_ctr(c, st));
    CKS(c, c->key.grow(c, (uint64_t)n, st));
    uint64_t tag;
    CKS(c, next_epoch(c, tag));
    CK(c, c->cand_slot.ensure((size_t)n * 4, 0, st));
    probe_list_kernel<IDENT_KEY><<<nblk(n), TILE, 0, st>>>(ck, n, c->key.as<uint64_t>(), c->key.units, tag, c->cand_slot.as<uint32_t>(), c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    c->key.occ += c->h_ctr->n_new;  // before the error check: a reset clears a partial insert too
    if (c->h_ctr->error) return fail(c, SPL_E_TABLE_FULL, "spl_dedup: probe overflow (table full)");
    const int64_t n_new = (int64_t)c->h_ctr->n_new;
    c->occupied += n_new;
    *n_out = n_new;
    if (n_new == 0) return SPL_OK;
    CK(c, c->tmp_rec.ensure((size_t)n_new * 32, 0, st));
    const unsigned nt = nblk(n, TILE * 32);
    CKS(c, prep_status(c, 0, nt, st));
    CKS(c, reset_ticket(c, 0, st));
    resolve_kernel<SRC_LIST, false><<<nt, TILE, sizeof(ResolveSmem), st>>>(
        nullptr, 0, c->d_tabs, c->d_takes_idx, c->d_takes_edges, nullptr, (uint32_t)n, c->key.as<uint64_t>(),
        c->cand_slot.as<uint32_t>(), ck, ca, 0, 0, c->tmp_rec.as<Rec>(), nullptr, usrc, 0, 0, c->luts,
        c->status[0].as<uint64_t>(), c->d_ctr, 0);
    unpack_rec_kernel<<<nblk(n_new), TILE, 0, st>>>(c->tmp_rec.as<Rec>(), n_new, uk, ua, nullptr);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaStreamSynchronize(st));
    return SPL_OK;
}

int32_t spl_add_formula(spl_ctx *c, const spl_formula *f, int32_t *id) {
    if (!c || !f || !id) return fail(c, SPL_E_INVALID, "spl_add_formula: null argument");
    if (const char *why = formula_error(*f)) return fail(c, SPL_E_INVALID, "spl_add_formula: %s", why);
    if (c->n_forms >= SPL_MAX_FORMULAS)
        return fail(c, SPL_E_CAPACITY, "spl_add_formula: a context holds at most %d formulas", (int)SPL_MAX_FORMULAS);
    // the (feature, exponent) pairs without a table yet; -0.0 + 0.0 == +0.0 keys both zeros alike
    const auto pair_of = [](int feat, double e) {
        const double z = e + 0.0;
        uint64_t bits;
        memcpy(&bits, &z, 8);
        return std::make_pair(feat, bits);
    };
    const auto find = [&](const std::pair<int, uint64_t> &k) -> double * {
        for (auto &t : c->pow_tabs)
            if (t.first == k) return t.second;
        return nullptr;
    };
    std::vector<std::pair<int, uint64_t>> fresh;
    uint64_t fresh_bytes = 0;
    for (int i = 0; i < f->n_terms; ++i)
        for (int j = 0; j < f->term[i].n_factors; ++j) {
            const auto k = pair_of(f->term[i].feature[j], f->term[i].exponent[j]);
            if (find(k) || std::find(fresh.begin(), fresh.end(), k) != fresh.end()) continue;
            fresh.push_back(k);
            fresh_bytes += 8ull * (formula_feature_max(k.first) + 1);
        }
    if (c->pow_bytes + fresh_bytes > SPL_FORMULA_TABLE_BYTES)
        return fail(c, SPL_E_CAPACITY, "spl_add_formula: the power tables of a context take at most %llu bytes (%llu in use, %llu more needed)",
                    (unsigned long long)SPL_FORMULA_TABLE_BYTES, (unsigned long long)c->pow_bytes, (unsigned long long)fresh_bytes);
    CK(c, enter_device(c));
    if (!c->d_forms) {
        CK(c, cudaMalloc(&c->d_forms, sizeof(FormDev) * SPL_MAX_FORMULAS));
    }
    for (const auto &k : fresh) {
        double e;
        memcpy(&e, &k.second, 8);
        const std::vector<double> t = formula_pow_table(k.first, e);
        double *d = nullptr;
        CK(c, cudaMalloc(&d, t.size() * 8));
        c->pow_tabs.emplace_back(k, d);
        c->pow_bytes += t.size() * 8;
        CK(c, cudaMemcpy(d, t.data(), t.size() * 8, cudaMemcpyHostToDevice));
        c->h2d_bytes += (long long)t.size() * 8;
    }
    FormDev F{};
    F.nt = f->n_terms;
    for (int i = 0; i < f->n_terms; ++i) {
        F.t[i].coef = f->term[i].coef;
        F.t[i].nf = f->term[i].n_factors;
        for (int j = 0; j < f->term[i].n_factors; ++j) {
            F.t[i].f[j].feat = f->term[i].feature[j];
            F.t[i].f[j].pw = find(pair_of(f->term[i].feature[j], f->term[i].exponent[j]));
        }
    }
    CK(c, cudaMemcpy(c->d_forms + c->n_forms, &F, sizeof F, cudaMemcpyHostToDevice));
    CK(c, cudaStreamSynchronize(nullptr));  // the pageable copies have landed before any later launch reads them
    c->h2d_bytes += (long long)sizeof F;
    *id = SPL_H_FORMULA_BASE + c->n_forms++;
    return SPL_OK;
}

int32_t spl_score(spl_ctx *c, int32_t heuristic, int32_t noise, const spl_key *keys, const uint64_t *aux, int64_t n,
                  double *scores, void *stream) {
    if (!c || n < 0) return fail(c, SPL_E_INVALID, "spl_score: bad arguments");
    CKS(c, check_heuristic(c, "spl_score", heuristic));
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    if (is_formula_id(heuristic)) score_kernel<true><<<nblk(n), TILE, 0, st>>>(keys, aux, n, heuristic, noise, c->luts, scores, c->d_forms);
    else score_kernel<false><<<nblk(n), TILE, 0, st>>>(keys, aux, n, heuristic, noise, c->luts, scores, nullptr);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_topk(spl_ctx *c, const double *scores, const spl_key *keys, int64_t n, int64_t k, int32_t tie_policy,
                 int64_t *out_idx, int64_t *n_out, void *stream) {
    if (!c || !n_out || n < 0 || n >= (1ll << 32) || k < 0) return fail(c, SPL_E_INVALID, "spl_topk: bad arguments");
    if (tie_policy != SPL_TIE_STABLE && tie_policy != SPL_TIE_KEY) return fail(c, SPL_E_INVALID, "spl_topk: unknown tie policy %d", tie_policy);
    if (tie_policy == SPL_TIE_KEY && !keys) return fail(c, SPL_E_INVALID, "spl_topk: SPL_TIE_KEY needs keys");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0 || k == 0) return SPL_OK;
    CKS(c, zero_ctr(c, st));
    CK(c, c->sk.ensure((size_t)n * 8, 0, st));
    flip_scores_kernel<<<nblk(n), TILE, 0, st>>>(scores, n, c->sk.as<uint64_t>(), c->d_ctr);
    ++c->launches;
    CKS(c, read_ctr(c, st));
    int which = 0;
    int64_t kept = 0;
    const uint64_t smin = c->h_ctr->sk_min, smax = c->h_ctr->sk_max;
    const Rec *recs = nullptr;
    if (tie_policy == SPL_TIE_KEY) {
        CK(c, c->tmp_rec.ensure((size_t)n * 32, 0, st));
        pack_rec_kernel<<<nblk(n), TILE, 0, st>>>(keys, nullptr, n, c->tmp_rec.as<Rec>());
        ++c->launches;
        recs = c->tmp_rec.as<Rec>();
    }
    CKS(c, run_cut_sort(c, c->sk.as<uint64_t>(), recs, n, k, smin, smax, CutMode{tie_policy == SPL_TIE_KEY ? TIES_KEY : TIES_ARRIVAL},
                        &which, &kept, st));
    idx_widen_kernel<<<nblk(kept), TILE, 0, st>>>(c->idx[which].as<uint32_t>(), kept, out_idx);
    ++c->launches;
    CK(c, cudaGetLastError());
    CK(c, cudaStreamSynchronize(st));
    *n_out = kept;
    return SPL_OK;
}

// ---- multi-GPU building blocks ----------------------------------------------------------------
// Per-owner counts from the digit-major scanned histogram in c->matrix2 (nt tiles per digit): owner g's candidates start
// at digit g, tile 0, and the last owner's end at n.  read_owner_starts queues the reads of the first n_read starts (the
// sort paths read n_ranks + 1); owner_counts takes the differences once the caller has synchronised the stream.
static int read_owner_starts(spl_ctx *c, unsigned nt, int n_read, std::vector<uint32_t> &start, cudaStream_t st) {
    start.resize(n_read);
    for (int g = 0; g < n_read; ++g)
        CK(c, cudaMemcpyAsync(&start[g], c->matrix2.as<uint32_t>() + (size_t)g * nt, 4, cudaMemcpyDeviceToHost, st));
    c->d2h_bytes += 4 * n_read;
    return SPL_OK;
}
static void owner_counts(const std::vector<uint32_t> &start, int n_ranks, int64_t n, int64_t *counts_host) {
    for (int g = 0; g < n_ranks; ++g) counts_host[g] = (g + 1 < n_ranks ? start[g + 1] : (uint32_t)n) - start[g];
}

int32_t spl_owner_partition(spl_ctx *c, const spl_key *keys, int64_t n, int32_t n_ranks, int64_t *perm, int64_t *counts_host,
                            void *stream) {
    if (!c || !counts_host || n < 0 || n >= (1ll << 32) || n_ranks < 1 || n_ranks > 256)
        return fail(c, SPL_E_INVALID, "spl_owner_partition: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    for (int g = 0; g < n_ranks; ++g) counts_host[g] = 0;
    if (n == 0) return SPL_OK;
    for (int b = 0; b < 2; ++b) {
        CK(c, c->y[b].ensure((size_t)n * 8 + 8, 0, st));
        CK(c, c->idx[b].ensure((size_t)n * 4 + 4, 0, st));
    }
    owner_kernel<<<nblk(n), TILE, 0, st>>>(keys, n, (uint32_t)n_ranks, c->y[0].as<uint64_t>(), c->idx[0].as<uint32_t>());
    ++c->launches;
    const unsigned nt = nblk(n, SORT_TILE);
    const size_t msz = (size_t)SORT_BINS * nt;
    CK(c, c->matrix.ensure(msz * 4, 0, st));
    CK(c, c->matrix2.ensure(msz * 4, 0, st));
    CKS(c, sort_pass(c, 0, 0, c->y[0].as<uint64_t>(), n, 0, nt, msz, st));  // one stable pass: digit = owner
    idx_widen_kernel<<<nblk(n), TILE, 0, st>>>(c->idx[1].as<uint32_t>(), n, perm);
    ++c->launches;
    std::vector<uint32_t> start;
    CKS(c, read_owner_starts(c, nt, n_ranks + 1, start, st));
    CK(c, cudaStreamSynchronize(st));
    owner_counts(start, n_ranks, n, counts_host);
    return SPL_OK;
}

// ---- row-based variants used by the sharded driver: rows are 32-byte records {lo, hi, aux, link}
int32_t spl_expand_rows(spl_ctx *c, const void *front_rows, int64_t n, int64_t rank_base, void *out_rows, int64_t cap,
                        int64_t *n_out, void *stream) {
    if (!c || !n_out || n < 0 || n > (16ll << 20)) return fail(c, SPL_E_INVALID, "spl_expand_rows: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0) return SPL_OK;
    CKS(c, zero_ctr(c, st));
    CKS(c, run_count(c, reinterpret_cast<const Rec *>(front_rows), n, st));
    const int64_t total = (int64_t)c->h_ctr->total_cands;
    *n_out = total;
    if (total > cap) return fail(c, SPL_E_CAPACITY, "spl_expand_rows: %lld successors, capacity %lld", (long long)total, (long long)cap);
    if (total == 0) return SPL_OK;
    expand_kernel<MODE_LIST, IDENT_KEY><<<nblk(n), TILE, sizeof(ExpandSmem2), st>>>(
        reinterpret_cast<const Rec *>(front_rows), n, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(),
        (uint32_t)total, nullptr, 0, 0, nullptr, reinterpret_cast<Rec *>(out_rows), rank_base, c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_route_keys(spl_ctx *c, const void *cand_rows, int64_t n, int32_t n_ranks, spl_key *send_keys, int64_t *counts_host,
                       void *stream) {
    if (!c || !counts_host || n < 0 || n >= (1ll << 32) || n_ranks < 1 || n_ranks > 255)
        return fail(c, SPL_E_INVALID, "spl_route_keys: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    for (int g = 0; g < n_ranks; ++g) counts_host[g] = 0;
    c->route_n = n;
    if (n == 0) return SPL_OK;
    for (int b = 0; b < 2; ++b) {
        CK(c, c->y[b].ensure((size_t)n * 8 + 8, 0, st));
        CK(c, c->idx[b].ensure((size_t)n * 4 + 4, 0, st));
    }
    const Rec *rows = reinterpret_cast<const Rec *>(cand_rows);
    if (n_ranks <= 32) {  // two kernels: per-tile owner histogram -> scan -> stable scatter of the keys
        const unsigned nt = nblk(n, PART_TILE);
        const size_t msz = (size_t)n_ranks * nt;
        CK(c, c->matrix.ensure(msz * 4 + 4, 0, st));
        CK(c, c->matrix2.ensure(msz * 4 + 4, 0, st));
        owner_hist_kernel<<<nt, TILE, 0, st>>>(rows, n, (uint32_t)n_ranks, c->matrix.as<uint32_t>(), nt);
        const unsigned st_tiles = nblk((int64_t)msz, TILE * SCAN_ITEMS);
        CKS(c, prep_status(c, 1, st_tiles, st));
        CKS(c, reset_ticket(c, 2, st));
        scan_u32_kernel<<<st_tiles, TILE, 0, st>>>(c->matrix.as<uint32_t>(), c->matrix2.as<uint32_t>(), (int64_t)msz,
                                                    c->status[1].as<uint64_t>(), c->d_ctr, 2);
        owner_scatter_kernel<<<nt, TILE, 0, st>>>(rows, n, (uint32_t)n_ranks, c->matrix2.as<uint32_t>(), nt, send_keys,
                                                   c->idx[1].as<uint32_t>());
        c->launches += 3;
        CK(c, cudaGetLastError());
        std::vector<uint32_t> start;
        CKS(c, read_owner_starts(c, nt, n_ranks, start, st));
        CK(c, cudaStreamSynchronize(st));
        owner_counts(start, n_ranks, n, counts_host);
        return SPL_OK;
    }
    owner_rows_kernel<<<nblk(n), TILE, 0, st>>>(rows, n, (uint32_t)n_ranks, c->y[0].as<uint64_t>(), c->idx[0].as<uint32_t>());
    ++c->launches;
    const unsigned nt = nblk(n, SORT_TILE);
    const size_t msz = (size_t)SORT_BINS * nt;
    CK(c, c->matrix.ensure(msz * 4, 0, st));
    CK(c, c->matrix2.ensure(msz * 4, 0, st));
    CKS(c, sort_pass(c, 0, 0, c->y[0].as<uint64_t>(), n, 0, nt, msz, st));  // stable: digit = owner; perm stays in idx[1]
    gather_keys_kernel<<<nblk(n), TILE, 0, st>>>(rows, c->idx[1].as<uint32_t>(), n, send_keys);
    ++c->launches;
    std::vector<uint32_t> start;
    CKS(c, read_owner_starts(c, nt, n_ranks + 1, start, st));
    CK(c, cudaStreamSynchronize(st));
    owner_counts(start, n_ranks, n, counts_host);
    return SPL_OK;
}

int32_t spl_score_rows(spl_ctx *c, int32_t heuristic, int32_t noise, const void *rows, int64_t n, double *scores,
                       const uint8_t *draws, void *stream) {
    if (!c || n < 0 || (noise == SPL_NOISE_EXTERNAL && !draws)) return fail(c, SPL_E_INVALID, "spl_score_rows: bad arguments");
    CKS(c, check_heuristic(c, "spl_score_rows", heuristic));
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    if (is_formula_id(heuristic))
        score_rows_kernel<true><<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const Rec *>(rows), n, heuristic, noise, c->luts, scores, draws,
                                                          c->d_forms);
    else
        score_rows_kernel<false><<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const Rec *>(rows), n, heuristic, noise, c->luts, scores, draws,
                                                           nullptr);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_dtopk_begin(spl_ctx *c, const double *scores, const spl_key *keys, int64_t n, uint64_t *sk_min_host,
                        uint64_t *sk_max_host, void *stream) {
    if (!c || !sk_min_host || !sk_max_host || n < 0 || n >= (1ll << 32)) return fail(c, SPL_E_INVALID, "spl_dtopk_begin: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    c->dtopk_n = n;
    c->dtopk_recs = false;
    *sk_min_host = ~0ull;
    *sk_max_host = 0;
    if (n == 0) return SPL_OK;
    CKS(c, zero_ctr(c, st));
    CK(c, c->sk.ensure((size_t)n * 8, 0, st));
    flip_scores_kernel<<<nblk(n), TILE, 0, st>>>(scores, n, c->sk.as<uint64_t>(), c->d_ctr);
    ++c->launches;
    if (keys) {  // the caller's key array must stay alive until spl_dtopk_cut
        c->dtopk_keys = reinterpret_cast<const uint64_t *>(keys);
        c->dtopk_recs = true;
    }
    CKS(c, read_ctr(c, st));
    *sk_min_host = c->h_ctr->sk_min;
    *sk_max_host = c->h_ctr->sk_max;
    return SPL_OK;
}

int32_t spl_dtopk_hist(spl_ctx *c, int32_t word, int32_t shift, int32_t bits, int32_t first, uint64_t sk_min_global,
                       uint32_t **hist_dev_out, void *stream) {
    if (!c || !hist_dev_out || word < 0 || word > 2 || bits < 1 || bits > SEL_BITS) return fail(c, SPL_E_INVALID, "spl_dtopk_hist: bad arguments");
    if (word > 0 && !c->dtopk_recs && c->dtopk_n) return fail(c, SPL_E_STATE, "spl_dtopk_hist: key passes need keys in spl_dtopk_begin");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    const int64_t n = c->dtopk_n;
    *hist_dev_out = c->d_hist;
    if (n == 0) return SPL_OK;
    const unsigned grid = std::min<unsigned>(nblk(n), 148 * 8);
    const uint64_t *sk = c->sk.as<uint64_t>();
    const uint64_t *kb = c->dtopk_keys;
    if (word == 0) sel_hist_kernel<0><<<grid, TILE, 0, st>>>(sk, kb, 2, n, sk_min_global, shift, bits, first, c->d_sel, c->d_hist);
    else if (word == 1) sel_hist_kernel<1><<<grid, TILE, 0, st>>>(sk, kb, 2, n, sk_min_global, shift, bits, first, c->d_sel, c->d_hist);
    else sel_hist_kernel<2><<<grid, TILE, 0, st>>>(sk, kb, 2, n, sk_min_global, shift, bits, first, c->d_sel, c->d_hist);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_dtopk_pick(spl_ctx *c, int32_t word, int32_t shift, int32_t first, int32_t init_k, int64_t k, void *stream) {
    if (!c) return SPL_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    sel_pick_kernel<<<1, 1024, 0, st>>>(c->d_hist, word, shift, first, init_k, (uint64_t)k, c->d_sel);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_dtopk_get(spl_ctx *c, uint64_t state_host[6], void *stream) {
    if (!c || !state_host) return SPL_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    CK(c, cudaMemcpyAsync(c->h_sel, c->d_sel, sizeof(SelState), cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    c->d2h_bytes += sizeof(SelState);
    memcpy(state_host, c->h_sel, 6 * sizeof(uint64_t));  // the six fields of the ABI; rank_t is internal
    return SPL_OK;
}

int32_t spl_dtopk_set(spl_ctx *c, const uint64_t state_host[6], void *stream) {
    if (!c || !state_host) return SPL_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    memcpy(c->h_sel, state_host, 6 * sizeof(uint64_t));
    c->h_sel->rank_t = ~0ull;
    CK(c, cudaMemcpyAsync(c->d_sel, c->h_sel, sizeof(SelState), cudaMemcpyHostToDevice, st));
    CK(c, cudaStreamSynchronize(st));
    c->h2d_bytes += sizeof(SelState);
    return SPL_OK;
}

int32_t spl_dtopk_cut(spl_ctx *c, int32_t tie_policy, int32_t keep_all, int32_t all_ties, uint64_t sk_min_global,
                      uint64_t sk_max_global, int64_t *out_idx, uint64_t *out_y, uint64_t *out_klo, uint64_t *out_khi,
                      int64_t *kept_host, void *stream) {
    if (!c || !kept_host) return SPL_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    const int64_t n = c->dtopk_n;
    *kept_host = 0;
    if (n == 0) return SPL_OK;
    CutMode mode;
    if (tie_policy == SPL_TIE_KEY) mode.ties = TIES_KEY;
    else if (tie_policy == SPL_TIE_KEY_ORDERED) mode.ties = TIES_KEY_ORDERED;
    if (mode.by_key() && !c->dtopk_recs) return fail(c, SPL_E_STATE, "spl_dtopk_cut: det policy needs keys in spl_dtopk_begin");
    int which = 0;
    int64_t kept = 0;
    CKS(c, do_cut_sort(c, c->sk.as<uint64_t>(), c->dtopk_keys, 2, n, n, keep_all, all_ties, sk_min_global, sk_max_global,
                       mode, 0, &which, &kept, st));
    if (kept) {
        idx_widen_kernel<<<nblk(kept), TILE, 0, st>>>(c->idx[which].as<uint32_t>(), kept, out_idx);
        ++c->launches;
        if (out_y) CK(c, cudaMemcpyAsync(out_y, c->y[which].p, (size_t)kept * 8, cudaMemcpyDeviceToDevice, st));
        if (mode.by_key() && out_klo) CK(c, cudaMemcpyAsync(out_klo, c->kl[which].p, (size_t)kept * 8, cudaMemcpyDeviceToDevice, st));
        if (mode.by_key() && out_khi) CK(c, cudaMemcpyAsync(out_khi, c->kh[which].p, (size_t)kept * 8, cudaMemcpyDeviceToDevice, st));
        CK(c, cudaGetLastError());
        CK(c, cudaStreamSynchronize(st));
    }
    *kept_host = kept;
    return SPL_OK;
}

int32_t spl_count_less(spl_ctx *c, int32_t words, int32_t inclusive, const uint64_t *ay, const uint64_t *akl,
                       const uint64_t *akh, int64_t na, const uint64_t *by, const uint64_t *bkl, const uint64_t *bkh,
                       int64_t nb, int64_t *out, int32_t accumulate, int32_t sorted_a, void *stream) {
    if (!c || (words != 1 && words != 3) || na < 0 || nb < 0) return fail(c, SPL_E_INVALID, "spl_count_less: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (na == 0) return SPL_OK;
    count_less_kernel<<<nblk(na), TILE, 0, st>>>(words, inclusive, ay, akl, akh, na, by, bkl, bkh, nb, out, accumulate, sorted_a);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ fused solver
// A pooled link column for `bytes`: the smallest pooled buffer that holds them, else the largest (it is regrown with
// 1/16 headroom -- queue lengths wobble by a fraction of a percent from level to level and from rank to rank, and
// every regrowth is a cudaMalloc plus a device-synchronising cudaFree in the middle of a level).
static DevBuf *take_link_buf(spl_ctx *c, size_t bytes) {
    if (c->pool_links.empty()) return new DevBuf();
    size_t best = c->pool_links.size(), big = 0;
    for (size_t i = 0; i < c->pool_links.size(); ++i) {
        const size_t cap = c->pool_links[i]->cap;
        if (cap >= bytes && (best == c->pool_links.size() || cap < c->pool_links[best]->cap)) best = i;
        if (cap > c->pool_links[big]->cap) big = i;
    }
    const size_t pick = best != c->pool_links.size() ? best : big;
    DevBuf *b = c->pool_links[pick];
    c->pool_links.erase(c->pool_links.begin() + (long)pick);
    return b;
}
static size_t link_bytes(int64_t n) { return (size_t)n * 8 + (size_t)n / 2; }

// Parent-link columns (src/solver.py:459-464 walks them back from the goal): one per level, 8 B per queue entry.  Past
// spl_set_link_budget's device budget the oldest columns move to pinned host memory (SURVEY.md 8(f).2); the path walk
// reads a spilled column in place.
struct LinkCols {
    std::vector<DevBuf *> dev;      // per level (pool-owned buffers)
    std::vector<uint64_t *> host;   // per level: pinned copy once spilled, else nullptr
    std::vector<int64_t> n;         // per level: entries
    size_t next_spill = 0;          // levels below this one are on the host
    ~LinkCols() { for (uint64_t *h : host) if (h) cudaFreeHost(h); }
    void push(DevBuf *b, int64_t cnt) { dev.push_back(b); host.push_back(nullptr); n.push_back(cnt); }
    // one entry, wherever the column lives
    cudaError_t read(int level, int64_t i, uint64_t *out) const {
        if (host[level]) { *out = host[level][i]; return cudaSuccess; }
        return cudaMemcpy(out, dev[level]->as<uint64_t>() + i, 8, cudaMemcpyDeviceToHost);
    }
    // spill oldest-first until the device-resident columns fit `budget` bytes (the newest column stays on the device)
    cudaError_t spill(uint64_t budget, uint64_t *moved, cudaStream_t st) {
        if (!budget) return cudaSuccess;
        uint64_t resident = 0;
        for (size_t l = next_spill; l < dev.size(); ++l) resident += (uint64_t)n[l] * 8;
        while (resident > budget && next_spill + 1 < dev.size()) {
            const size_t l = next_spill++;
            const size_t bytes = (size_t)n[l] * 8;
            if (!bytes) continue;
            cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&host[l]), bytes);
            if (e != cudaSuccess) { host[l] = nullptr; return e; }
            e = cudaMemcpyAsync(host[l], dev[l]->p, bytes, cudaMemcpyDeviceToHost, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return e;
            dev[l]->release();  // the memory goes back to the device, not to the column pool
            resident -= bytes;
            *moved += bytes;
        }
        return cudaSuccess;
    }
};

// What a solver holds while it is open: the queue buffers, lent by its context (the last solve's, so that their memory
// is reused), and per level the queue's parent links and, on the card-set-sharded driver, its global ranks.
struct SolverBufs {
    spl_ctx *c;
    int keep_links = 1;
    DevBuf front, uniq, grank;
    LinkCols links, ranks;
    explicit SolverBufs(spl_ctx *ctx) : c(ctx) {
        front.swap(c->pool_front);
        uniq.swap(c->pool_uniq);
        grank.swap(c->pool_grank);
        std::sort(c->pool_links.begin(), c->pool_links.end(), [](DevBuf *a, DevBuf *b) { return a->cap > b->cap; });
    }
    ~SolverBufs() {
        if (c->active == this) c->active = nullptr;
        c->pool_front.swap(front);  // keep the big buffers for the next solve on this context
        c->pool_uniq.swap(uniq);
        c->pool_grank.swap(grank);
        for (auto *b : links.dev) c->pool_links.push_back(b);
        for (auto *b : ranks.dev) c->pool_links.push_back(b);
    }
    void activate() { c->active = this; }
};

// Append the columns of a level whose queue is front[0..n): the parent links (from 96-byte realistic records when
// `realistic`) and, with `with_ranks`, the global ranks in grank.  Then spill the oldest columns to pinned host memory
// past the context's link budget, which the columns of a level share evenly.
static int save_links(SolverBufs *s, int64_t n, bool realistic, bool with_ranks, cudaStream_t st) {
    spl_ctx *c = s->c;
    const bool keep = s->keep_links && n > 0;
    const size_t need = keep ? (size_t)n * 8 : 0;
    const int ncols = with_ranks ? 2 : 1;
    LinkCols *cols[2] = {&s->links, &s->ranks};
    DevBuf *buf[2] = {nullptr, nullptr};
    for (int i = 0; i < ncols; ++i) {
        buf[i] = take_link_buf(c, need);  // columns of earlier solves on this context
        cols[i]->push(buf[i], s->keep_links ? n : 0);
    }
    if (!keep) return SPL_OK;
    for (int i = 0; i < ncols; ++i)
        if (buf[i]->cap < need) CK(c, buf[i]->ensure(link_bytes(n), 0, st));
    if (realistic)
        r_links_kernel<<<nblk(n), TILE, 0, st>>>(s->front.as<RRec>(), n, buf[0]->as<uint64_t>());
    else
        unpack_rec_kernel<<<nblk(n), TILE, 0, st>>>(s->front.as<Rec>(), n, nullptr, nullptr, buf[0]->as<uint64_t>());
    ++c->launches;
    if (with_ranks) CK(c, cudaMemcpyAsync(buf[1]->p, s->grank.p, need, cudaMemcpyDeviceToDevice, st));
    CK(c, cudaGetLastError());
    uint64_t moved = 0;
    for (int i = 0; i < ncols; ++i) CK(c, cols[i]->spill(c->link_budget / ncols, &moved, st));
    c->d2h_bytes += moved;
    c->spilled_bytes += moved;
    return SPL_OK;
}

// The formulation of a solver's levels (DESIGN.md 3), and with it its visited table.
enum LevelKind {
    KEY_TABLE,  // expand + dedup against the key table, in chunks of parents
    GROUPED,    // beam search on the card-set-grouped level (spl_m2.cuh), visited set in the node table
    REALISTIC,  // realistic mode: materialised 96-byte successors, exact-key table
    REALISTIC_BATCH,  // realistic mode, many games in lockstep: game-major queues, (game, exact key) table
    SPEEDRUN_BATCH,   // speedrun mode, many games in lockstep: game-major 32-byte queues, (game, key) table (spl_sbatch.cuh)
};
static const VisitTable &visited_table(const spl_ctx *c, LevelKind kind) {
    return kind == KEY_TABLE ? c->key : kind == GROUPED ? c->nodes : kind == REALISTIC ? c->rtab
         : kind == REALISTIC_BATCH ? c->rbtab : c->sbtab;
}

// What a batched solver keeps beside the common queue buffers (spl_rbatch_*, spl_realistic.cuh; spl_sbatch_*,
// spl_sbatch.cuh): the games' configs (RConfigDev or SGame) and roots, the queue's game-major offsets (on the device for
// the kernels, on the host per level for the line walk), the per-game counters, and the game column of the candidates
// and of the winners.
struct RBatch {
    int B = 0;
    std::vector<int64_t> beam;
    std::vector<spl_rgame_info> info;          // per game: the counters of the last level it took part in
    std::vector<int64_t> final_rank;           // per ended game: rank of its last state in the queue of info.level
    std::vector<std::vector<int64_t>> seg_at;  // per level: the queue offsets of the games (B + 1)
    DevBuf cfg, roots, seg, gctr, cand_game, uniq_game, scratch, lines;
};

struct spl_solver : SolverBufs {
    int goal = 15, use_h = 0, heuristic = 0, tie = 0, noise = 0;
    bool form = false;  // batch: some beam game scores with a formula (sb_score_kernel<true>)
    LevelKind kind = KEY_TABLE;
    spl_rconfig rcfg{};
    // external-noise mode: the level is split in two calls (expand+dedup | score+cut)
    bool pending = false;
    int64_t pend_n = 0, pend_uniq = 0;
    spl_level_info pend_info{};
    int64_t beam = 300000;
    int64_t n_front = 0;
    int level = 0;
    bool ended = false;
    int64_t goal_rank = -1;
    std::unique_ptr<RBatch> rb;  // REALISTIC_BATCH and SPEEDRUN_BATCH only
    explicit spl_solver(spl_ctx *ctx) : SolverBufs(ctx) {}
};

// What the expand + dedup half of a level leaves for the cut: n_uniq states in the first n_slots elements of s->uniq
// (n_slots > n_uniq: the grouped level leaves unused slots) and, where scores were computed on the way, their range.
struct LevelExpand {
    int64_t n_uniq = 0, n_slots = 0, generated = 0;
    uint64_t sk_min = ~0ull, sk_max = 0;
};

// ------------------------------------------------------------------ card-set-grouped level (spl_m2.cuh)
// One-sweep stable LSD sort (spl_m2.cuh 2b) of k[*cur][0..n) by bits lo_bit .. lo_bit + nbits - 1, ping-ponging between
// k[0] / k[1]; with a payload column (pl != nullptr) the pairs move together.  n < OS_MAX_ITEMS.
static int onesweep_sort(spl_ctx *c, uint64_t *const k[2], uint32_t *const pl[2], int64_t n, int lo_bit, int nbits, int *cur, cudaStream_t st) {
    const int passes = (nbits + OS_BITS - 1) / OS_BITS;
    if (n <= 1 || passes <= 0) return SPL_OK;
    if (passes > OS_MAX_PASSES || n >= OS_MAX_ITEMS) return fail(c, SPL_E_INVALID, "internal: one-sweep sort of %lld values, %d bits", (long long)n, nbits);
    const unsigned snt = nblk(n, SORT_TILE);
    const size_t status_bytes = (size_t)snt * OS_BINS * 4;
    CK(c, c->os_hist.ensure(OS_MAX_PASSES * OS_BINS * 4, 0, st));
    CK(c, c->os_status.ensure(status_bytes, 0, st));
    CK(c, cudaMemsetAsync(c->os_hist.p, 0, (size_t)passes * OS_BINS * 4, st));
    os_hist_kernel<<<std::min<unsigned>(148 * 8, nblk(n)), TILE, (size_t)passes * OS_BINS * 4, st>>>(k[*cur], n, lo_bit, passes, c->os_hist.as<uint32_t>());
    os_base_kernel<<<passes, OS_BINS, 0, st>>>(c->os_hist.as<uint32_t>());
    c->launches += 2;
    for (int p = 0; p < passes; ++p) {
        CK(c, cudaMemsetAsync(c->os_status.p, 0, status_bytes, st));
        CKS(c, reset_ticket(c, 2, st));
        if (pl)
            os_scatter_kernel<true><<<snt, TILE, sizeof(OsSmem), st>>>(k[*cur], pl[*cur], n, lo_bit + p * OS_BITS, c->os_hist.as<uint32_t>() + p * OS_BINS,
                                                                       c->os_status.as<uint32_t>(), c->d_ctr, 2, k[*cur ^ 1], pl[*cur ^ 1]);
        else
            os_scatter_kernel<false><<<snt, TILE, offsetof(OsSmem, stage_p), st>>>(k[*cur], nullptr, n, lo_bit + p * OS_BITS,
                                                                                   c->os_hist.as<uint32_t>() + p * OS_BINS,
                                                                                   c->os_status.as<uint32_t>(), c->d_ctr, 2, k[*cur ^ 1], nullptr);
        ++c->launches;
        CK(c, cudaGetLastError());
        *cur ^= 1;
    }
    return SPL_OK;
}

// Stable sort of the round's packed items by their key bits ITEM_KEY_LO..63: three one-sweep passes of 10-bit digits
// (rounds below 2^30 items), else 8-bit LSD passes with per-pass histogram + scan.
static int sort_items(spl_ctx *c, int64_t n_items, int *cur, cudaStream_t st) {
    const unsigned snt = nblk(n_items, SORT_TILE);
    if (n_items < OS_MAX_ITEMS) {
        uint64_t *const k[2] = {c->y[0].as<uint64_t>(), c->y[1].as<uint64_t>()};
        return onesweep_sort(c, k, nullptr, n_items, ITEM_KEY_LO, 64 - ITEM_KEY_LO, cur, st);
    }
    const int lo_bit = ITEM_KEY_LO;
    const size_t msz = (size_t)SORT_BINS * snt;
    CK(c, c->matrix.ensure(msz * 4, 0, st));
    CK(c, c->matrix2.ensure(msz * 4, 0, st));
    const unsigned st_tiles = nblk((int64_t)msz, TILE * SCAN_ITEMS);
    if (n_items > 1)
        for (int shift = lo_bit; shift < 64; shift += SORT_BITS) {
            sort_hist_kernel<<<snt, TILE, 0, st>>>(c->y[*cur].as<uint64_t>(), n_items, shift, c->matrix.as<uint32_t>(), snt);
            CKS(c, prep_status(c, 1, st_tiles, st));
            CKS(c, reset_ticket(c, 2, st));
            scan_u32_kernel<<<st_tiles, TILE, 0, st>>>(c->matrix.as<uint32_t>(), c->matrix2.as<uint32_t>(), (int64_t)msz,
                                                        c->status[1].as<uint64_t>(), c->d_ctr, 2);
            psort_scatter_kernel<<<snt, TILE, 0, st>>>(c->y[*cur].as<uint64_t>(), n_items, shift, c->matrix2.as<uint32_t>(), snt,
                                                        c->y[*cur ^ 1].as<uint64_t>());
            c->launches += 3;
            CK(c, cudaGetLastError());
            *cur ^= 1;
        }
    return SPL_OK;
}

// One round of a grouped level after its fan-out, the same on one GPU and on the card-set-sharded driver.
struct GroupRound {
    const Rec *front = nullptr;      // the round's parents
    const Rec *brec = nullptr;       // the buy records this rank received (sharded; one GPU: rebuilt from front)
    int64_t np = 0, n_items = 0;     // parents; items packed in c->y[0], the parents' first
    uint64_t n_cands = 0;            // candidates (gem takes + buy records): the most winners the round can have
    int64_t rank_base = 0;           // queue rank of front[0] (one GPU) ...
    const uint64_t *grank = nullptr; // ... or the parents' global ranks (sharded)
    bool unordered = false;          // the records arrive in no particular order (sharded): the warp kernel sorts them
    DevBuf *out = nullptr;           // winners go to out / c->sk from slot out_base on
    int64_t out_base = 0;
    int heuristic = 0, noise = 0, level = 0;
};
struct RoundTimes { float sort, prep, thread, warp, cta; };

  // CUDA-event ms: item sort + runs, node table + buffers, the kernels

// Sort the round's items by card-set hash, find the runs of equal key, then deduplicate every run against the node
// table: thread kernel over all runs, then the warp kernel and the CTA kernel over the runs each one queued.  The caller
// has zeroed the counters; they hold the round's on return.
static int group_round(spl_ctx *c, const GroupRound &R, int64_t *n_new_out, RoundTimes *t, cudaStream_t st) {
    CK(c, cudaEventRecord(c->ev[1], st));
    int cur = 0;
    CKS(c, sort_items(c, R.n_items, &cur, st));
    const unsigned rt = nblk(R.n_items, TILE * RUN_ITEMS);  // runs of equal key + candidate-weight prefix
    CK(c, c->run_start.ensure((size_t)R.n_items * 4 + 8, 0, st));
    CK(c, c->run_wpre.ensure((size_t)R.n_items * 4 + 8, 0, st));
    CKS(c, prep_status(c, 1, rt, st));
    CKS(c, prep_status(c, 2, rt, st));
    CKS(c, reset_ticket(c, 1, st));
    m2_runs_kernel<<<rt, TILE, 0, st>>>(c->y[cur].as<uint64_t>(), R.n_items, (uint32_t)R.np, c->ntk8.as<uint8_t>(), c->run_start.as<uint32_t>(),
                                         c->run_wpre.as<uint32_t>(), c->status[1].as<uint64_t>(), c->status[2].as<uint64_t>(), c->d_ctr, 1);
    ++c->launches;
    CK(c, cudaGetLastError());
    CK(c, cudaEventRecord(c->ev[2], st));
    CKS(c, read_ctr(c, st));
    const uint64_t n_runs = c->h_ctr->n_runs;
    // every run holds at least one card set; more than one only when two sets share the 30 sorted hash bits
    CKS(c, c->nodes.grow(c, n_runs + n_runs / 8 + 64, st));
    CK(c, c->cls_list.ensure((size_t)n_runs * 8 + 16, 0, st));
    const size_t n_out = (size_t)R.out_base + (size_t)R.n_cands;
    CK(c, R.out->ensure(n_out * 32, (size_t)R.out_base * 32, st));
    CK(c, c->sk.ensure(n_out * 8, (size_t)R.out_base * 8, st));
    GroupArgs A;
    A.front = R.front; A.brec = R.brec; A.iv = c->y[cur].as<uint64_t>();
    A.run_start = c->run_start.as<uint32_t>(); A.run_wpre = c->run_wpre.as<uint32_t>();
    A.np = (uint32_t)R.np; A.rank_base = R.rank_base; A.grank = R.grank; A.unordered = R.unordered;
    A.warp_max = R.unordered ? std::min<uint32_t>(BIG_W, BSORT_MAX) : BIG_W;  // the warp kernel sorts at most BSORT_MAX records of a run itself
    A.tabs = c->d_tabs; A.takes_idx = c->d_takes_idx; A.takes_pk = c->d_takes_pk; A.take_rows = c->d_take_rows; A.gemrank = c->d_gemrank; A.rankgems = c->d_rankgems;
    A.nodes = c->nodes.as<uint64_t>(); A.nn = c->nodes.units; A.out = R.out->as<Rec>(); A.out_sk = c->sk.as<uint64_t>(); A.out_base = (uint64_t)R.out_base;
    for (int k = 0; k < NUM_CLS; ++k) A.cls_list[k] = nullptr;
    A.cls_list[CLS_WARP] = c->cls_list.as<uint32_t>();
    A.cls_list[CLS_CTA] = c->cls_list.as<uint32_t>() + n_runs;
    A.h = R.heuristic; A.noise_mode = R.noise; A.L = c->luts; A.ctr = c->d_ctr;
    CK(c, cudaEventRecord(c->ev[3], st));
    if (R.unordered) m2_group_tiny_kernel<true><<<nblk((int64_t)n_runs), TILE, 0, st>>>(A, (uint32_t)n_runs);
    else m2_group_tiny_kernel<false><<<nblk((int64_t)n_runs), TILE, 0, st>>>(A, (uint32_t)n_runs);
    CK(c, cudaEventRecord(c->ev[4], st));
    CKS(c, reset_ticket(c, 2, st));  // the warp kernel draws its runs from ticket 2
    if (R.unordered) m2_group_warp_kernel<true><<<148 * SPL_WARP_CTAS, TILE, sizeof(WarpSmem), st>>>(A);
    else m2_group_warp_kernel<false><<<148 * SPL_WARP_CTAS, TILE, offsetof(WarpSmem, bsort), st>>>(A);  // no sort area
    CK(c, cudaEventRecord(c->ev[5], st));
    if (R.unordered) m2_group_big_kernel<true><<<148 * 5, TILE, sizeof(BigSmem), st>>>(A);
    else m2_group_big_kernel<false><<<148 * 5, TILE, sizeof(BigSmem), st>>>(A);
    c->launches += 3;
    CK(c, cudaGetLastError());
    CK(c, cudaEventRecord(c->ev[6], st));
    CKS(c, read_ctr(c, st));
    const Counters &h = *c->h_ctr;
    cudaEventElapsedTime(&t->sort, c->ev[1], c->ev[2]);
    cudaEventElapsedTime(&t->prep, c->ev[2], c->ev[3]);
    cudaEventElapsedTime(&t->thread, c->ev[3], c->ev[4]);
    cudaEventElapsedTime(&t->warp, c->ev[4], c->ev[5]);
    cudaEventElapsedTime(&t->cta, c->ev[5], c->ev[6]);
    if (getenv("SPL_DEBUG"))
        fprintf(stderr, "[grouped] L%d np=%lld items=%lld runs=%llu cls=%u/%u/%u new_nodes=%u winners=%llu | sort+runs %.2f prep %.2f thread %.2f warp %.2f cta %.2f ms | nodes %llu/%llu\n",
                R.level, (long long)R.np, (long long)R.n_items, (unsigned long long)n_runs,
                (unsigned)(n_runs - h.n_cls[CLS_WARP] - h.n_cls[CLS_CTA]), h.n_cls[CLS_WARP], h.n_cls[CLS_CTA], h.n_new_nodes,
                (unsigned long long)h.n_emitted, t->sort, t->prep, t->thread, t->warp, t->cta, (unsigned long long)c->nodes.occ,
                (unsigned long long)c->nodes.units);
    c->nodes.occ += h.n_new_nodes;  // before the error checks: a reset clears a partial insert too
    if (h.error == 3)
        return fail(c, SPL_E_CUDA, "level %d: more than %d card sets share one 30-bit sort key in a run of the warp kernel (or more than %d in one of the CTA kernel)",
                    R.level, MAX_SETS + 1, BIG_DONE + 1);
    if (h.error)
        return fail(c, SPL_E_TABLE_FULL, "card-set table full during level %d (device error %u; %llu slots, max_node_bytes=%llu)", R.level,
                    h.error, (unsigned long long)c->nodes.units, (unsigned long long)c->nodes.max_bytes);
    // A formula search runs the dedup kernels unchanged: they score its winners as they score an unknown id, with
    // `simple`, and this pass replaces those score keys and their range by the formula's (the caller reads sk_min /
    // sk_max from h_ctr).  The formula evaluator inside the register-bound warp and CTA kernels would spill.
    if (is_formula_id(R.heuristic) && h.n_emitted) {
        const unsigned long long range0[2] = {~0ull, 0ull};
        static_assert(offsetof(Counters, sk_max) == offsetof(Counters, sk_min) + 8, "sk_min, sk_max adjacent");
        CK(c, cudaMemcpyAsync(&c->d_ctr->sk_min, range0, sizeof range0, cudaMemcpyHostToDevice, st));
        c->h2d_bytes += sizeof range0;
        score_rec_kernel<<<nblk((int64_t)h.n_emitted), TILE, 0, st>>>(R.out->as<Rec>() + R.out_base, nullptr, (int64_t)h.n_emitted,
                                                                      c->d_forms + (R.heuristic - SPL_H_FORMULA_BASE), R.noise,
                                                                      c->sk.as<uint64_t>() + R.out_base, c->d_ctr);
        ++c->launches;
        CK(c, cudaGetLastError());
        CKS(c, read_ctr(c, st));
    }
    c->occupied += h.n_emitted;
    *n_new_out = (int64_t)h.n_emitted;
    return SPL_OK;
}

// expand + dedup (+ score) of the whole queue `front[0..n)` in rounds of parents; winners are appended to
// s->uniq / c->sk in no particular order (their link words carry the arrival order)
static int grouped_expand(spl_solver *s, int64_t n, LevelExpand *x, float ms[6], cudaStream_t st) {
    spl_ctx *c = s->c;
    const Rec *front = s->front.as<Rec>();
    const int64_t chunk = c->chunk_user ? (int64_t)c->chunk_parents : (int64_t)MAX_CHUNK_PARENTS;
    int64_t n_uniq = 0, n_slots = 0, generated = 0;
    uint64_t sk_min = ~0ull, sk_max = 0;
    for (int64_t p0 = 0; p0 < n; p0 += chunk) {
        const int64_t np = std::min<int64_t>(chunk, n - p0);
        const unsigned nt = nblk(np);
        // fan-out: buys offsets, take counts, sort keys of the parents
        CKS(c, zero_ctr(c, st));
        CK(c, cudaEventRecord(c->ev[0], st));
        CK(c, c->boff2.ensure((size_t)np * 4 + 4, 0, st));
        CK(c, c->ntk8.ensure((size_t)np + 8, 0, st));
        // items of the round = parents + buys (packed: hash half << 32 | item id); the array is sized for the parents
        // first and grown (contents kept) once the buys are counted
        CK(c, c->y[0].ensure((size_t)np * 8 + 8, 0, st));
        CKS(c, prep_status(c, 0, nt, st));
        m2_count_kernel<<<nt, TILE, 0, st>>>(front + p0, np, c->d_tabs, c->d_takes_idx, c->boff2.as<uint32_t>(),
                                              c->y[0].as<uint64_t>(), c->ntk8.as<uint8_t>(), c->status[0].as<uint64_t>(), c->d_ctr, 0);
        ++c->launches;
        CK(c, cudaGetLastError());
        CKS(c, read_ctr(c, st));
        const uint64_t n_takes = c->h_ctr->total_cands, n_buys = c->h_ctr->n_buys, total = n_takes + n_buys;
        generated += (int64_t)total;
        if (total == 0) continue;
        const int64_t n_items = np + (int64_t)n_buys;
        if (total >= 0xFFFFFFFFull || (uint64_t)n_items >= 0xFFFFFFFFull)
            return fail(c, SPL_E_INVALID, "round produced %llu candidates (>= 2^32): lower spl_config.chunk_parents", (unsigned long long)total);
        CK(c, c->y[0].ensure((size_t)n_items * 8 + 8, (size_t)np * 8, st));
        CK(c, c->y[1].ensure((size_t)n_items * 8 + 8, 0, st));
        if (n_buys) {
            m2_buys_kernel<<<nt, TILE, sizeof(BuySmem), st>>>(front + p0, np, c->d_tabs, c->d_takes_idx, c->boff2.as<uint32_t>(),
                                                               c->y[0].as<uint64_t>());
            ++c->launches;
            CK(c, cudaGetLastError());
        }
        GroupRound R;
        R.front = front + p0; R.np = np; R.n_items = n_items; R.n_cands = total; R.rank_base = p0;
        R.out = &s->uniq; R.out_base = n_slots; R.heuristic = s->heuristic; R.noise = s->noise; R.level = s->level;
        int64_t n_new = 0;
        RoundTimes t;
        CKS(c, group_round(c, R, &n_new, &t, st));
        if (n_new) { sk_min = std::min<uint64_t>(sk_min, c->h_ctr->sk_min); sk_max = std::max<uint64_t>(sk_max, c->h_ctr->sk_max); }
        n_uniq += n_new;
        n_slots += n_new;  // dense output
        float t_count;
        cudaEventElapsedTime(&t_count, c->ev[0], c->ev[1]);
        ms[0] += t_count;                        // fan-out + buy items
        ms[2] += t.sort;                         // item sort + runs (grouping)
        ms[1] += t.thread + t.warp + t.cta;      // per-run dedup + emit + score (the dominant stage)
        ms[5] += t.warp;                         // ... of which the warp kernel
    }
    *x = LevelExpand{n_uniq, n_slots, generated, sk_min, sk_max};
    return SPL_OK;
}

// ------------------------------------------------------------------ solver create
// The realistic tables and the batch tables (rtab, rbtab, sbtab) are allocated on first use, sized by the caller's
// table_slots.  They do not use the key table: a large, empty one gives its memory back first.
static int open_rtable(spl_ctx *c, cudaStream_t st, VisitTable &t) {
    if (t.p) return SPL_OK;
    if (c->key.occ == 0 && c->key.units > (1ull << 16)) CK(c, c->key.alloc(buckets_for(1ull << 12), st));
    uint64_t nb = std::max<uint64_t>(c->rslots_hint ? c->rslots_hint : (1ull << 16), 1024);
    nb = std::min<uint64_t>(nb, t.max_bytes / t.d.unit_bytes);
    CK(c, t.alloc(nb, st));
    return SPL_OK;
}
static int open_rtable(spl_ctx *c, cudaStream_t st) { return open_rtable(c, st, c->rtab); }

// What every solver create shares: clear the visited sets, upload the n level-0 rows (`row_bytes` each: a 32-byte Rec
// or a 96-byte realistic record) and, on the card-set-sharded driver, the root's global rank 0; register the rows in
// the visited table of the level kind (trail = {row: None for row in rows}); save the first link columns, synchronise
// and go live.  With n = 0 (a sharded rank that does not own the root's card set) the queue starts empty.  Realistic
// mode and the sharded driver start from one root (n <= 1), the batched realistic search from one root per game.  On
// error `s` is deleted.
template <class S>
static int open_solver(S *s, LevelKind kind, const void *rows, int64_t n, size_t row_bytes, bool sharded, const char *sync_msg,
                       S **out) {
    spl_ctx *c = s->c;
    const cudaStream_t st = 0;
    const int rc = [&]() -> int {
        CKS(c, reset_visited(c, st));
        if (n) {
            const uint64_t zero = 0;
            const size_t bytes = (size_t)n * row_bytes;
            cudaError_t e = s->front.ensure(bytes, 0, st);
            if (e == cudaSuccess) e = cudaMemcpyAsync(s->front.p, rows, bytes, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess && sharded) e = s->grank.ensure(8, 0, st);
            if (e == cudaSuccess && sharded) e = cudaMemcpyAsync(s->grank.p, &zero, 8, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaStreamSynchronize(st);
            c->h2d_bytes += bytes + (sharded ? 8 : 0);
            if (e != cudaSuccess) return fail(c, SPL_E_CUDA, "root upload: %s", cudaGetErrorString(e));
            CKS(c, zero_ctr(c, st));
            uint64_t tag = 0;
            if (kind == KEY_TABLE) {
                CKS(c, c->key.grow(c, (uint64_t)n, st));
                CKS(c, next_epoch(c, tag));
                if (c->cand_slot.ensure((size_t)n * 4, 0, st) != cudaSuccess) return fail(c, SPL_E_NOMEM, "cand_slot alloc");
                const spl_key *k = s->front.template as<spl_key>();  // a Rec starts with its key
                constexpr int REC_KEYS = sizeof(Rec) / sizeof(spl_key);
                if (c->identity == IDENT_PYHASH)
                    probe_list_kernel<IDENT_PYHASH, REC_KEYS><<<nblk(n), TILE, 0, st>>>(k, n, c->key.as<uint64_t>(), c->key.units, tag,
                                                                              c->cand_slot.as<uint32_t>(), c->d_ctr);
                else
                    probe_list_kernel<IDENT_KEY, REC_KEYS><<<nblk(n), TILE, 0, st>>>(k, n, c->key.as<uint64_t>(), c->key.units, tag,
                                                                           c->cand_slot.as<uint32_t>(), c->d_ctr);
                c->key.occ = (uint64_t)n;
            } else if (kind == GROUPED) {
                CKS(c, c->nodes.grow(c, (uint64_t)n, st));
                m2_root_kernel<<<nblk(n), TILE, 0, st>>>(c->nodes.as<uint64_t>(), c->nodes.units, s->front.template as<Rec>(), n,
                                                         c->d_gemrank, c->d_ctr);
                c->nodes.occ = (uint64_t)n;  // card sets registered, at most: only the table's load factor reads it
            } else if (kind == REALISTIC) {
                if (c->cand_slot.ensure(4, 0, st) != cudaSuccess) return fail(c, SPL_E_NOMEM, "realistic scratch alloc");
                CKS(c, open_rtable(c, st));
                CKS(c, c->rtab.grow(c, 1, st));
                if (c->rtab.clear(st) != cudaSuccess) return fail(c, SPL_E_CUDA, "realistic table reset failed");  // forget the previous search
                CKS(c, next_epoch(c, tag));
                r_probe_kernel<<<1, TILE, 0, st>>>(s->front.template as<RRec>(), 1, c->rcfg.as<RConfigDev>(), c->rtab.as<RBucket>(),
                                                    c->rtab.units, tag, c->cand_slot.as<uint32_t>(), c->d_ctr);
                c->rtab.occ = 1;
            } else if constexpr (std::is_same_v<S, spl_solver>) {  // the batches: one root per game, rb->cand_game = 0 .. n - 1
                VisitTable &t = kind == REALISTIC_BATCH ? c->rbtab : c->sbtab;
                if (c->cand_slot.ensure((size_t)n * 4, 0, st) != cudaSuccess) return fail(c, SPL_E_NOMEM, "batch scratch alloc");
                CKS(c, open_rtable(c, st, t));
                CKS(c, t.grow(c, (uint64_t)n, st));
                if (t.clear(st) != cudaSuccess) return fail(c, SPL_E_CUDA, "batch table reset failed");
                CKS(c, next_epoch(c, tag));
                CKS(c, zero_ctr(c, st));  // after the table's growth
                RBatch &R = *s->rb;
                unsigned long long *n_new_game = R.gctr.as<unsigned long long>() + 2 * R.B;
                if (kind == REALISTIC_BATCH)
                    rb_probe_kernel<<<nblk(n), TILE, 0, st>>>(s->front.template as<RRec>(), R.cand_game.as<uint32_t>(), n,
                                                              R.cfg.as<RConfigDev>(), t.as<RBucket>(), t.units, tag,
                                                              c->cand_slot.as<uint32_t>(), c->d_ctr, n_new_game);
                else
                    sb_probe_kernel<<<nblk(n), TILE, 0, st>>>(s->front.template as<Rec>(), R.cand_game.as<uint32_t>(), n,
                                                              t.as<SBucket>(), t.units, tag, c->cand_slot.as<uint32_t>(), c->d_ctr,
                                                              n_new_game);
                t.occ = (uint64_t)n;
            }
            ++c->launches;
            CK(c, cudaGetLastError());
            c->occupied = (uint64_t)n;
        }
        CKS(c, save_links(s, n, kind == REALISTIC || kind == REALISTIC_BATCH, sharded, st));
        if (cudaStreamSynchronize(st) != cudaSuccess) return fail(c, SPL_E_CUDA, "%s", sync_msg);
        return SPL_OK;
    }();
    if (rc != SPL_OK) { delete s; return rc; }
    s->activate();
    *out = s;
    return SPL_OK;
}

// ------------------------------------------------------------------ sharded grouped level (spl_shard.cuh)
// One spl_gsolver per rank.  The host (Python, torch.distributed) issues the collectives between these calls:
//   level:  spl_gs_goal -> all-reduce MIN
//           per round: spl_gs_round_begin (-> per-destination record counts) -> all-gather of the counts ->
//                      spl_gs_round_buys (records into the send buffer) -> all-to-all -> spl_gs_round_group
//           cut:    spl_gs_dict -> all-gather -> spl_gs_threshold [-> spl_gs_tie_begin, (spl_gs_tie_hist -> all-reduce
//                      -> spl_gs_tie_pick) x passes] -> spl_gs_cut (local survivors, sorted by their sort word)
//           ranks:  sample sort of the sort words across ranks (spl_gs_partition / spl_gs_rank_sort + all-to-all) ->
//                   spl_gs_adopt (next queue = survivors with their global ranks)
struct spl_gsolver : SolverBufs {
    int rank = 0, world = 1, goal = 15, heuristic = 0, noise = 0;
    int64_t beam = 0;
    int64_t n_local = 0, n_global = 1;
    int level = 0;
    // round
    int64_t r_p0 = 0, r_np = 0;
    uint64_t r_takes = 0, r_buys = 0;
    int64_t counts[MAX_RANKS]{};
    // level accumulators
    int64_t n_uniq = 0, generated = 0;
    float ms[4] = {0, 0, 0, 0};  // CUDA-event time of: item sort + runs, thread kernel, table warp kernel, CTA kernel
    // cut
    int lt = 0, cut_cur = 0;
    int64_t kept_local = 0;
    explicit spl_gsolver(spl_ctx *ctx) : SolverBufs(ctx) {}
};

extern "C" {

int32_t spl_gs_create(spl_ctx *c, int32_t rank, int32_t world, const spl_key *root_key, uint64_t root_aux, int32_t goal,
                      int32_t heuristic, int64_t beam, int32_t noise, int32_t keep_links, spl_gsolver **out) {
    if (!c || !root_key || !out || world < 1 || world > MAX_RANKS || rank < 0 || rank >= world || beam < 1)
        return fail(c, SPL_E_INVALID, "spl_gs_create: bad arguments (1 <= world <= %d)", MAX_RANKS);
    if (noise != SPL_NOISE_CONST && noise != SPL_NOISE_HASH) return fail(c, SPL_E_INVALID, "spl_gs_create: noise must be const or hash");
    CKS(c, check_heuristic(c, "spl_gs_create", heuristic));
    NO_LIVE_SOLVER(c, "spl_gs_create");
    CK(c, enter_device(c));
    spl_gsolver *s = new spl_gsolver(c);
    s->rank = rank; s->world = world; s->goal = goal; s->heuristic = heuristic; s->beam = beam; s->noise = noise;
    s->keep_links = keep_links;
    const Rec r{root_key->lo, root_key->hi & HI_KEY_MASK, root_aux, ~0ull};
    uint64_t m0, m1;
    mask_words(r.lo, r.hi, m0, m1);
    const bool owner = (int)owner_of_mask(m0, m1, (uint32_t)world) == rank;  // the root lives on the rank that owns its card set
    s->n_local = owner ? 1 : 0;
    return open_solver(s, GROUPED, &r, owner ? 1 : 0, 32, true, "spl_gs_create: sync failed", out);
}

int32_t spl_gs_destroy(spl_gsolver *s) {
    if (s) { cudaSetDevice(s->c->device); cudaDeviceSynchronize(); delete s; }
    return SPL_OK;
}

// first local queue state with pts >= goal -> its GLOBAL rank (INT64_MAX: none); also the local queue length
int32_t spl_gs_goal(spl_gsolver *s, int64_t *rank_host, int64_t *n_local_host, void *stream) {
    if (!s || !rank_host || !n_local_host) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *rank_host = 0x7fffffffffffffffll;
    *n_local_host = s->n_local;
    s->n_uniq = 0;
    s->generated = 0;
    s->ms[0] = s->ms[1] = s->ms[2] = s->ms[3] = 0;
    if (s->n_local == 0) return SPL_OK;
    CKS(c, zero_ctr(c, st));
    goal_kernel<<<nblk(s->n_local), TILE, 0, st>>>(s->front.as<Rec>(), s->n_local, s->goal, c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    if (c->h_ctr->goal_rank != 0x7fffffffffffffffll) {
        uint64_t g = 0;
        CK(c, cudaMemcpyAsync(&g, s->grank.as<uint64_t>() + c->h_ctr->goal_rank, 8, cudaMemcpyDeviceToHost, st));
        CK(c, cudaStreamSynchronize(st));
        c->d2h_bytes += 8;
        *rank_host = (int64_t)g;
    }
    return SPL_OK;
}

// first local index whose global rank is >= r (the local queue is ascending in global rank)
static int gs_lower(spl_gsolver *s, int64_t r, int64_t *idx, cudaStream_t st) {
    spl_ctx *c = s->c;
    int64_t lo = 0, hi = s->n_local;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        uint64_t v = 0;
        CK(c, cudaMemcpyAsync(&v, s->grank.as<uint64_t>() + mid, 8, cudaMemcpyDeviceToHost, st));
        CK(c, cudaStreamSynchronize(st));
        c->d2h_bytes += 8;
        if ((int64_t)v < r) lo = mid + 1; else hi = mid;
    }
    *idx = lo;
    return SPL_OK;
}

// round = the local parents whose global rank is in [rank_lo, rank_hi): fan-out, sort keys, and the number of buy
// records this rank will send to every rank (counts_host[world])
int32_t spl_gs_round_begin(spl_gsolver *s, int64_t rank_lo, int64_t rank_hi, int64_t *counts_host, int64_t *n_parents_host,
                           void *stream) {
    if (!s || !counts_host || !n_parents_host) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    int64_t p0 = 0, p1 = s->n_local;
    if (rank_lo > 0) CKS(c, gs_lower(s, rank_lo, &p0, st));
    if (rank_hi < s->n_global) CKS(c, gs_lower(s, rank_hi, &p1, st));
    const int64_t np = p1 - p0;
    s->r_p0 = p0; s->r_np = np; s->r_takes = s->r_buys = 0;
    for (int g = 0; g < s->world; ++g) counts_host[g] = s->counts[g] = 0;
    *n_parents_host = np;
    if (np == 0) return SPL_OK;
    if (np >= (1ll << 31)) return fail(c, SPL_E_INVALID, "round of %lld parents: use smaller rank windows", (long long)np);
    CKS(c, zero_ctr(c, st));
    CK(c, cudaMemsetAsync(c->d_dest, 0, 2 * MAX_RANKS * 8, st));
    CK(c, c->ntk8.ensure((size_t)np + 8, 0, st));
    CK(c, c->y[0].ensure((size_t)np * 8 + 8, 0, st));
    gs_count_kernel<<<nblk(np), TILE, 0, st>>>(s->front.as<Rec>() + p0, np, c->d_tabs, c->d_takes_idx, c->y[0].as<uint64_t>(),
                                                c->ntk8.as<uint8_t>(), (uint32_t)s->world, c->d_dest, c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    unsigned long long h_dest[MAX_RANKS];
    CK(c, cudaMemcpyAsync(h_dest, c->d_dest, MAX_RANKS * 8, cudaMemcpyDeviceToHost, st));
    CKS(c, read_ctr(c, st));
    c->d2h_bytes += MAX_RANKS * 8;
    s->r_takes = c->h_ctr->total_cands;
    s->r_buys = c->h_ctr->n_buys;
    uint64_t sum = 0;
    for (int g = 0; g < s->world; ++g) { counts_host[g] = s->counts[g] = (int64_t)h_dest[g]; sum += h_dest[g]; }
    if (sum != s->r_buys) return fail(c, SPL_E_CUDA, "internal: destination counts %llu != buys %llu", (unsigned long long)sum, (unsigned long long)s->r_buys);
    s->generated += (int64_t)(s->r_takes + s->r_buys);
    return SPL_OK;
}

// the round's buy records into send_dev: destination d owns [sum(counts[0..d)), +counts[d])
// the round's buy records, destination d's at dst[d] + (0 .. counts[d]) in no particular order
static int gs_route(spl_gsolver *s, void *const *dst, cudaStream_t st) {
    spl_ctx *c = s->c;
    unsigned long long h[2 * MAX_RANKS] = {0};  // cursors (relative to each destination's base), then the bases
    for (int g = 0; g < s->world; ++g) h[MAX_RANKS + g] = (unsigned long long)(uintptr_t)dst[g];
    CK(c, cudaMemcpyAsync(c->d_dest + MAX_RANKS, h, sizeof(h), cudaMemcpyHostToDevice, st));
    CK(c, cudaStreamSynchronize(st));  // h is a stack array
    c->h2d_bytes += sizeof(h);
    gs_buys_route_kernel<<<nblk(s->r_np), TILE, sizeof(RouteSmem), st>>>(
        s->front.as<Rec>() + s->r_p0, s->r_np, s->grank.as<uint64_t>() + s->r_p0, c->d_tabs, c->d_takes_idx, (uint32_t)s->world,
        reinterpret_cast<Rec *const *>(c->d_dest + 2 * MAX_RANKS), c->d_dest + MAX_RANKS);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_gs_round_buys(spl_gsolver *s, void *send_dev, void *stream) {
    if (!s) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (s->r_np == 0 || s->r_buys == 0) return SPL_OK;
    if (!send_dev) return fail(c, SPL_E_INVALID, "spl_gs_round_buys: null send buffer");
    void *dst[MAX_RANKS] = {nullptr};
    int64_t at = 0;
    for (int g = 0; g < s->world; ++g) { dst[g] = reinterpret_cast<Rec *>(send_dev) + at; at += s->counts[g]; }
    return gs_route(s, dst, st);
}

int32_t spl_gs_round_buys_peer(spl_gsolver *s, void *const *recv_dev_of_rank, const int64_t *offset_at_rank, void *stream) {
    if (!s || !recv_dev_of_rank || !offset_at_rank) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (s->r_np == 0 || s->r_buys == 0) return SPL_OK;
    void *dst[MAX_RANKS] = {nullptr};
    for (int g = 0; g < s->world; ++g) {
        if (s->counts[g] && (!recv_dev_of_rank[g] || offset_at_rank[g] < 0)) return fail(c, SPL_E_INVALID, "spl_gs_round_buys_peer: no buffer for rank %d", g);
        dst[g] = reinterpret_cast<Rec *>(recv_dev_of_rank[g]) + offset_at_rank[g];
    }
    return gs_route(s, dst, st);
}

// ---- device buffers other processes of this node can map (CUDA IPC): the receive side of spl_gs_round_buys_peer
int32_t spl_ipc_alloc(spl_ctx *c, uint64_t bytes, void **ptr_out, uint8_t handle_out[64]) {
    if (!c || !ptr_out || !handle_out || !bytes) return SPL_E_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "the ABI carries CUDA IPC handles as 64 bytes");
    CK(c, enter_device(c));
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(c, SPL_E_NOMEM, "spl_ipc_alloc: %llu bytes: %s", (unsigned long long)bytes, cudaGetErrorString(e)); }
    cudaIpcMemHandle_t h;
    e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); cudaGetLastError(); return fail(c, SPL_E_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e)); }
    memcpy(handle_out, &h, 64);
    *ptr_out = p;
    return SPL_OK;
}
int32_t spl_ipc_open(spl_ctx *c, const uint8_t handle[64], void **ptr_out) {
    if (!c || !handle || !ptr_out) return SPL_E_INVALID;
    CK(c, enter_device(c));
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    cudaError_t e = cudaIpcOpenMemHandle(ptr_out, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) { cudaGetLastError(); return fail(c, SPL_E_CUDA, "cudaIpcOpenMemHandle: %s", cudaGetErrorString(e)); }
    return SPL_OK;
}
int32_t spl_ipc_close(spl_ctx *c, void *ptr) {
    if (!c || !ptr) return SPL_E_INVALID;
    CK(c, enter_device(c));
    CK(c, cudaIpcCloseMemHandle(ptr));
    return SPL_OK;
}
int32_t spl_ipc_free(spl_ctx *c, void *ptr) {
    if (!c || !ptr) return SPL_E_INVALID;
    CK(c, enter_device(c));
    CK(c, cudaDeviceSynchronize());
    CK(c, cudaFree(ptr));
    return SPL_OK;
}

// owner side: the round's local parents + the n_recv records received for this rank -> sort by card set, per-run
// dedup against this rank's nodes, winners (+ scores) appended to the level's list
int32_t spl_gs_round_group(spl_gsolver *s, const void *recv_dev, int64_t n_recv, int64_t *n_new_host, void *stream) {
    if (!s || !n_new_host || n_recv < 0) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_new_host = 0;
    const int64_t np = s->r_np, n_items = np + n_recv;
    const uint64_t total = s->r_takes + (uint64_t)n_recv;
    if (total == 0) return SPL_OK;
    if (total >= 0xFFFFFFFFull || (uint64_t)n_items >= 0xFFFFFFFFull)
        return fail(c, SPL_E_INVALID, "round holds %llu candidates (>= 2^32): use smaller rank windows", (unsigned long long)total);
    CK(c, c->y[0].ensure((size_t)n_items * 8 + 8, (size_t)np * 8, st));
    CK(c, c->y[1].ensure((size_t)n_items * 8 + 8, 0, st));
    CKS(c, zero_ctr(c, st));  // a rank without parents in this round skipped the one in spl_gs_round_begin
    if (n_recv) {
        gs_recv_items_kernel<<<nblk(n_recv), TILE, 0, st>>>(reinterpret_cast<const Rec *>(recv_dev), n_recv, (uint32_t)np, c->y[0].as<uint64_t>());
        ++c->launches;
    }
    GroupRound R;
    R.front = s->front.as<Rec>() + s->r_p0; R.brec = reinterpret_cast<const Rec *>(recv_dev); R.np = np; R.n_items = n_items;
    R.n_cands = total; R.grank = s->grank.as<uint64_t>() + s->r_p0; R.unordered = true; R.out = &s->uniq; R.out_base = s->n_uniq;
    R.heuristic = s->heuristic; R.noise = s->noise; R.level = s->level;
    int64_t n_new = 0;
    RoundTimes t;
    CKS(c, group_round(c, R, &n_new, &t, st));
    s->ms[0] += t.sort + t.prep; s->ms[1] += t.thread; s->ms[2] += t.warp; s->ms[3] += t.cta;
    s->n_uniq += n_new;
    *n_new_host = n_new;
    return SPL_OK;
}

int32_t spl_gs_stage_ms(spl_gsolver *s, float ms_host[4]) {
    if (!s || !ms_host) return SPL_E_INVALID;
    for (int i = 0; i < 4; ++i) ms_host[i] = s->ms[i];
    return SPL_OK;
}

int32_t spl_gs_counters(spl_gsolver *s, int64_t *n_uniq_host, int64_t *generated_host, int64_t *visited_host) {
    if (!s) return SPL_E_INVALID;
    if (n_uniq_host) *n_uniq_host = s->n_uniq;
    if (generated_host) *generated_host = s->generated;
    if (visited_host) *visited_host = (int64_t)s->c->occupied;
    return SPL_OK;
}

// local dictionary of the level's scores (distinct score -> count); *dict_dev points at sizeof(ScoreDict) = *bytes
int32_t spl_gs_dict(spl_gsolver *s, void **dict_dev, int64_t *bytes, void *stream) {
    if (!s || !dict_dev || !bytes) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    CK(c, cudaMemsetAsync(c->d_dict->key, 0xFF, sizeof(c->d_dict->key), st));
    CK(c, cudaMemsetAsync(c->d_dict->cnt, 0, sizeof(ScoreDict) - sizeof(c->d_dict->key), st));
    if (s->n_uniq) {
        dict_build_kernel<<<std::min<unsigned>(nblk(s->n_uniq), 148 * 8), TILE, 0, st>>>(c->sk.as<uint64_t>(), s->n_uniq, c->d_dict);
        ++c->launches;
        CK(c, cudaGetLastError());
    }
    *dict_dev = c->d_dict;
    *bytes = (int64_t)sizeof(ScoreDict);
    return SPL_OK;
}

// all ranks' dictionaries (all-gathered, `world` x sizeof(ScoreDict)) -> global threshold for the k best of
// n_uniq_global states.  *need_ties_host = 1: the threshold score has more states than fit (split by arrival order)
int32_t spl_gs_threshold(spl_gsolver *s, const void *dicts_dev, int64_t k, int64_t n_uniq_global, int32_t *need_ties_host,
                         void *stream) {
    if (!s || !dicts_dev || !need_ties_host || k < 1) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    CK(c, cudaMemsetAsync(c->d_dict2->key, 0xFF, sizeof(c->d_dict2->key), st));
    CK(c, cudaMemsetAsync(c->d_dict2->cnt, 0, sizeof(ScoreDict) - sizeof(c->d_dict2->key), st));
    memset(c->h_sel, 0, sizeof(SelState));
    c->h_sel->rank_t = ~0ull;
    CK(c, cudaMemcpyAsync(c->d_sel, c->h_sel, sizeof(SelState), cudaMemcpyHostToDevice, st));
    gs_dict_merge_kernel<<<nblk((int64_t)s->world * DICT_CAP), TILE, 0, st>>>(reinterpret_cast<const ScoreDict *>(dicts_dev), s->world, c->d_dict2);
    dict_rank_kernel<<<1, 1024, 0, st>>>(c->d_dict2, (uint64_t)std::min(k, n_uniq_global), 0, c->d_sel);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(c->h_sel, c->d_sel, sizeof(SelState), cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    c->d2h_bytes += sizeof(SelState);
    if (c->h_sel->rank_t == ~0ull)
        return fail(c, SPL_E_CAPACITY, "the level has more than %d distinct scores: the dictionary cut does not apply", DICT_MAX);
    s->lt = 8 + bitlen((uint64_t)s->n_global);
    *need_ties_host = (n_uniq_global > k && c->h_sel->k_rem < c->h_sel->tie_count) ? 1 : 0;
    if (!*need_ties_host) c->h_sel->tie_count = 0;  // all ties are kept
    return SPL_OK;
}

// ties of the threshold score: collect their arrival words locally, then radix-select the quota-th one globally --
// the host all-reduces *hist_dev (2048 x uint32) between spl_gs_tie_hist and spl_gs_tie_pick; passes: shift = lt - 11,
// lt - 22, ... (bits = min(11, remaining))
int32_t spl_gs_tie_begin(spl_gsolver *s, int32_t *link_bits_host, void *stream) {
    if (!s || !link_bits_host) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *link_bits_host = s->lt;
    CK(c, c->rtmp.ensure((size_t)std::max<int64_t>(s->n_uniq, 1) * 8 + 8, 0, st));
    CK(c, cudaMemsetAsync(&c->d_ctr->n_ties, 0, 8, st));
    if (s->n_uniq) {
        tie_collect_kernel<<<std::min<unsigned>(nblk(s->n_uniq), 148 * 8), TILE, 0, st>>>(
            c->sk.as<uint64_t>(), reinterpret_cast<const uint64_t *>(s->uniq.p), 4, s->n_uniq, 0, c->d_sel, s->lt, c->rtmp.as<uint64_t>(), c->d_ctr);
        ++c->launches;
        CK(c, cudaGetLastError());
    }
    CKS(c, read_ctr(c, st));
    return SPL_OK;
}
int32_t spl_gs_tie_hist(spl_gsolver *s, int32_t shift, int32_t bits, int32_t first, uint32_t **hist_dev, void *stream) {
    if (!s || !hist_dev) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *hist_dev = c->d_hist;
    const int64_t ntie = (int64_t)c->h_ctr->n_ties;
    if (ntie) {
        sel_hist_kernel<3><<<std::min<unsigned>(nblk(ntie), 148 * 8), TILE, 0, st>>>(nullptr, c->rtmp.as<uint64_t>(), 1, ntie, 0, shift, bits, first,
                                                                                    c->d_sel, c->d_hist);
        ++c->launches;
        CK(c, cudaGetLastError());
    }
    return SPL_OK;
}
int32_t spl_gs_tie_pick(spl_gsolver *s, int32_t shift, int32_t first, void *stream) {
    if (!s) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    sel_pick_kernel<<<1, 1024, 0, st>>>(c->d_hist, 2, shift, first, 0, 0, c->d_sel);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

// local cut by the global threshold, then local sort by the sort word (score rank << link bits | link: ascending ==
// better first, and a total order over all ranks).  *y_sorted_dev: the kept_local sort words, ascending.
int32_t spl_gs_cut(spl_gsolver *s, int32_t have_tie_threshold, int64_t *kept_local_host, const uint64_t **y_sorted_dev, int32_t *y_bits_host,
                   void *stream) {
    if (!s || !kept_local_host || !y_sorted_dev || !y_bits_host) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    const int64_t n = s->n_uniq;
    const int nbits = s->lt + bitlen(c->h_sel->rank_t);
    *y_bits_host = nbits;
    *kept_local_host = s->kept_local = 0;
    *y_sorted_dev = nullptr;
    s->cut_cur = 0;
    if (n == 0) return SPL_OK;
    int cur = 0;
    int64_t kept = 0;
    CKS(c, cut_packed(c, c->sk.as<uint64_t>(), reinterpret_cast<const uint64_t *>(s->uniq.p), 4, n, n, 0, 0, have_tie_threshold ? 0 : 1,
                      c->d_dict2, s->lt, &cur, &kept, st));
    s->cut_cur = cur;
    *kept_local_host = s->kept_local = kept;
    *y_sorted_dev = c->y[cur].as<uint64_t>();
    return SPL_OK;
}

// lower bounds of n_probes ascending probes in the local sorted sort words (sample-sort partition)
int32_t spl_gs_partition(spl_gsolver *s, const uint64_t *probes_host, int32_t n_probes, int64_t *bounds_host, void *stream) {
    if (!s || n_probes < 0 || n_probes > 4 * MAX_RANKS) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n_probes == 0) return SPL_OK;
    CK(c, c->rtmp.ensure(16 * 4 * MAX_RANKS, 0, st));
    uint64_t *dp = c->rtmp.as<uint64_t>();
    int64_t *dout = reinterpret_cast<int64_t *>(dp + 4 * MAX_RANKS);
    CK(c, cudaMemcpyAsync(dp, probes_host, (size_t)n_probes * 8, cudaMemcpyHostToDevice, st));
    gs_lower_bound_kernel<<<1, 64, 0, st>>>(c->y[s->cut_cur].as<uint64_t>(), s->kept_local, dp, n_probes, dout);
    ++c->launches;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(bounds_host, dout, (size_t)n_probes * 8, cudaMemcpyDeviceToHost, st));
    CK(c, cudaStreamSynchronize(st));
    return SPL_OK;
}

// receiver side of the sample sort: n sort words (any order) -> ranks_out[i] = base + (number of words smaller than
// word i); the words of all ranks are pairwise distinct (they contain the arrival index)
int32_t spl_gs_rank_sort(spl_gsolver *s, const uint64_t *y_dev, int64_t n, int32_t y_bits, int64_t base, int64_t *ranks_out_dev, void *stream) {
    if (!s || n < 0) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    if (n >= OS_MAX_ITEMS) return fail(c, SPL_E_INVALID, "spl_gs_rank_sort: %lld sort words (limit 2^30 per rank)", (long long)n);
    // y[] / idx[] of the context hold the local survivors (spl_gs_cut): work in separate buffers
    CK(c, c->kl[0].ensure((size_t)n * 8 + 8, 0, st));
    CK(c, c->kl[1].ensure((size_t)n * 8 + 8, 0, st));
    CK(c, c->kh[0].ensure((size_t)n * 4 + 8, 0, st));
    CK(c, c->kh[1].ensure((size_t)n * 4 + 8, 0, st));
    CK(c, cudaMemcpyAsync(c->kl[0].p, y_dev, (size_t)n * 8, cudaMemcpyDeviceToDevice, st));
    gs_iota_kernel<<<nblk(n), TILE, 0, st>>>(c->kh[0].as<uint32_t>(), n);
    ++c->launches;
    int cur = 0;
    {
        uint64_t *const k[2] = {c->kl[0].as<uint64_t>(), c->kl[1].as<uint64_t>()};
        uint32_t *const pl[2] = {c->kh[0].as<uint32_t>(), c->kh[1].as<uint32_t>()};
        CKS(c, onesweep_sort(c, k, pl, n, 0, y_bits, &cur, st));
    }
    gs_scatter_ranks_kernel<<<nblk(n), TILE, 0, st>>>(c->kh[cur].as<uint32_t>(), n, base, ranks_out_dev);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

// next queue of this rank = its survivors in sort-word order (== ascending global rank) with the global ranks the
// sample sort assigned (granks_dev[i] for the i-th local survivor); n_global_next = queue length over all ranks
int32_t spl_gs_adopt(spl_gsolver *s, const int64_t *granks_dev, int64_t n_global_next, void *stream) {
    if (!s) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    const int64_t kept = s->kept_local;
    const bool dbg = getenv("SPL_DEBUG") != nullptr;
    if (dbg) CK(c, cudaEventRecord(c->ev[0], st));
    if (kept) {
        if (!granks_dev) return fail(c, SPL_E_INVALID, "spl_gs_adopt: null ranks");
        CK(c, s->front.ensure((size_t)kept * 32, 0, st));
        CK(c, s->grank.ensure((size_t)kept * 8, 0, st));
        gather_rec_kernel<<<nblk(kept), TILE, 0, st>>>(s->uniq.as<Rec>(), c->idx[s->cut_cur].as<uint32_t>(), kept, s->front.as<Rec>());
        ++c->launches;
        CK(c, cudaMemcpyAsync(s->grank.p, granks_dev, (size_t)kept * 8, cudaMemcpyDeviceToDevice, st));
        CK(c, cudaGetLastError());
    }
    s->n_local = kept;
    s->n_global = n_global_next;
    s->level += 1;
    if (dbg) CK(c, cudaEventRecord(c->ev[1], st));
    CKS(c, save_links(s, s->n_local, false, true, st));
    if (dbg) CK(c, cudaEventRecord(c->ev[2], st));
    CK(c, cudaStreamSynchronize(st));
    if (dbg) {
        float t1 = 0, t2 = 0;
        cudaEventElapsedTime(&t1, c->ev[0], c->ev[1]); cudaEventElapsedTime(&t2, c->ev[1], c->ev[2]);
        fprintf(stderr, "[gs r%d] adopt L%d kept=%lld gather %.2f links %.2f ms\n", s->rank, s->level, (long long)kept, t1, t2);
    }
    return SPL_OK;
}

// device view of the local queue: records (32 B each) and their global ranks
int32_t spl_gs_frontier(spl_gsolver *s, const void **recs_dev, const uint64_t **granks_dev, int64_t *n_local_host) {
    if (!s || !n_local_host) return SPL_E_INVALID;
    if (recs_dev) *recs_dev = s->front.p;
    if (granks_dev) *granks_dev = s->grank.as<uint64_t>();
    *n_local_host = s->n_local;
    return SPL_OK;
}

// link (parent rank << 8 | ordinal) of the state with global rank `grank` in the queue of `level`, if this rank holds it
int32_t spl_gs_link_at(spl_gsolver *s, int32_t level, int64_t grank, int32_t *found_host, uint64_t *link_host) {
    if (!s || !found_host || !link_host || level < 0 || level >= (int)s->ranks.dev.size()) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    if (!s->keep_links) return fail(c, SPL_E_STATE, "spl_gs_link_at: solver was created with keep_links = 0");
    CK(c, enter_device(c));
    *found_host = 0;
    *link_host = 0;
    const int64_t n = s->ranks.n[level];
    int64_t lo = 0, hi = n;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        uint64_t v = 0;
        CK(c, s->ranks.read(level, mid, &v));
        if ((int64_t)v < grank) lo = mid + 1; else hi = mid;
    }
    if (lo < n) {
        uint64_t v = 0;
        CK(c, s->ranks.read(level, lo, &v));
        if ((int64_t)v == grank) {
            CK(c, s->links.read(level, lo, link_host));
            *found_host = 1;
        }
    }
    return SPL_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ realistic mode host side
// the kernels' form of a config (checked)
static int make_rconfig(spl_ctx *c, const spl_rconfig *cfg, RConfigDev &h) {
    if (!cfg || cfg->num_players < 2 || cfg->num_players > 4 || cfg->gems_per_color < 1 || cfg->gems_per_color > 7)
        return fail(c, SPL_E_INVALID, "realistic config: num_players must be 2..4 and gems_per_color 1..7");
    const HostTables &T = host_tables();
    memset(&h, 0, sizeof h);
    h.P = cfg->num_players; h.target = cfg->target_points; h.gpc = cfg->gems_per_color; h.noise = cfg->noise;
    for (int t = 0; t < 3; ++t) {
        if (cfg->deck_len[t] < 0 || cfg->deck_len[t] > 40) return fail(c, SPL_E_INVALID, "realistic config: bad deck length");
        h.deck_len[t] = cfg->deck_len[t];
        memcpy(h.deck[t], cfg->deck[t], 40);
        for (int i = 0; i < cfg->deck_len[t]; ++i)
            if (cfg->deck[t][i] < SPL_NUM_CARDS) h.pos_of[cfg->deck[t][i]] = (uint8_t)i;
    }
    for (int i = 0; i < SPL_NUM_CARDS; ++i) {
        const int t = T.card_pt[i] == 0 ? 0 : T.card_pt[i] <= 2 ? 1 : 2;  // tiers by points, src/solver.py:102-104
        if (i < 64) { h.col_lo[T.card_bonus[i]] |= 1ull << i; h.pt_lo[T.card_pt[i]] |= 1ull << i; h.tier_lo[t] |= 1ull << i; }
        else { h.col_hi[T.card_bonus[i]] |= 1u << (i - 64); h.pt_hi[T.card_pt[i]] |= 1u << (i - 64); h.tier_hi[t] |= 1u << (i - 64); }
        h.card[i] = T.dev.card[i];
    }
    return SPL_OK;
}
static int upload_rconfig(spl_ctx *c, const spl_rconfig *cfg, cudaStream_t st) {
    RConfigDev h;
    CKS(c, make_rconfig(c, cfg, h));
    CK(c, c->rcfg.ensure(sizeof h, 0, st));
    c->rcfg_dirty = true;
    c->rcfg_have = false;
    CK(c, cudaMemcpyAsync(c->rcfg.p, &h, sizeof h, cudaMemcpyHostToDevice, st));
    CK(c, cudaStreamSynchronize(st));  // h is a stack object
    c->h2d_bytes += sizeof h;
    c->rcfg_host = *cfg;
    c->rcfg_have = true;
    return SPL_OK;
}
// upload only when the device copy holds another config (the sharded driver passes the same one every round)
static int use_rconfig(spl_ctx *c, const spl_rconfig *cfg, cudaStream_t st) {
    if (cfg && c->rcfg_have && memcmp(&c->rcfg_host, cfg, sizeof *cfg) == 0) return SPL_OK;
    return upload_rconfig(c, cfg, st);
}

// count + scan of the successors of front[0..n): offsets in c->off, vis masks in c->rvmask, the count in *total (synchronises)
static int r_count_scan(spl_ctx *c, const RRec *front, int64_t n, int64_t *total, cudaStream_t st) {
    const unsigned nt = nblk(n);
    CK(c, c->off.ensure((size_t)n * 4 + 4, 0, st));
    CK(c, c->rvmask.ensure((size_t)n * 4 + 4, 0, st));
    CKS(c, zero_ctr(c, st));
    CKS(c, prep_status(c, 0, nt, st));
    r_count_scan_kernel<<<nt, TILE, 0, st>>>(front, n, c->rcfg.as<RConfigDev>(), c->off.as<uint32_t>(), c->rvmask.as<uint32_t>(),
                                              c->status[0].as<uint64_t>(), c->d_ctr, 0);
    ++c->launches;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    *total = (int64_t)c->h_ctr->total_cands;
    return SPL_OK;
}

// count + materialise the successors of front[0..n) into c->rcand
static int r_expand_all(spl_ctx *c, const RRec *front, int64_t n, int64_t rank_base, int64_t *total_out, cudaStream_t st) {
    CKS(c, r_count_scan(c, front, n, total_out, st));
    const int64_t total = *total_out;
    if (total == 0) return SPL_OK;
    CK(c, c->rcand.ensure((size_t)total * 96, 0, st));
    r_expand_kernel<<<nblk(n), TILE, 0, st>>>(front, n, c->rcfg.as<RConfigDev>(), c->off.as<uint32_t>(), c->rvmask.as<uint32_t>(),
                                               rank_base, c->rcand.as<RRec>());
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

// ---- row layer of the key-sharded driver, shared by speedrun (Rec, spl_*) and realistic (RRec, spl_r*) rows
// Owner side of a key-sharded round: first-arrival insert of a received key list (index = arrival) into the speedrun
// table (16-byte keys) or the realistic one (RKEY_WORDS-word keys), then one winner byte per key.
static int dedup_flags(spl_ctx *c, bool realistic, const void *keys, int64_t n, uint8_t *flags, cudaStream_t st) {
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    CKS(c, zero_ctr(c, st));
    if (realistic) CKS(c, open_rtable(c, st));
    VisitTable &t = realistic ? c->rtab : c->key;
    CKS(c, t.grow(c, (uint64_t)n, st));
    uint64_t tag;
    CKS(c, next_epoch(c, tag));
    CK(c, c->cand_slot.ensure((size_t)n * 4, 0, st));
    uint32_t *slot = c->cand_slot.as<uint32_t>();
    if (realistic) {
        CKS(c, zero_ctr(c, st));  // again after the table's growth, as realistic_expand does
        r_probe_keys_kernel<<<nblk(n), TILE, 0, st>>>(static_cast<const uint64_t *>(keys), n, t.as<RBucket>(), t.units, tag, slot, c->d_ctr);
        win_flags_kernel<<<nblk(n), TILE, 0, st>>>(slot, t.as<RBucket>(), n, flags);
    } else {
        probe_list_kernel<IDENT_KEY><<<nblk(n), TILE, 0, st>>>(static_cast<const spl_key *>(keys), n, t.as<uint64_t>(), t.units, tag, slot, c->d_ctr);
        win_flags_kernel<<<nblk(n), TILE, 0, st>>>(slot, t.as<uint64_t>(), n, flags);
    }
    c->launches += 2;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    t.occ += c->h_ctr->n_new;  // before the error check: a reset clears a partial insert too
    if (c->h_ctr->error && realistic)
        return fail(c, SPL_E_TABLE_FULL, "spl_rdedup_flags: probe overflow (realistic visited table full, %llu buckets)", (unsigned long long)t.units);
    if (c->h_ctr->error) return fail(c, SPL_E_TABLE_FULL, "spl_dedup_flags: probe overflow (table full)");
    if (!realistic) c->occupied += c->h_ctr->n_new;
    return SPL_OK;
}

// Source side of a key-sharded round: winner bytes in the send order of the route call this follows (route_n candidates,
// permutation perm; `what` is the SPL_E_STATE message) -> the winning rows in arrival order.
template <typename R>
static int compact_winners(spl_ctx *c, int64_t route_n, const uint32_t *perm, const char *what, const void *cand, int64_t n,
                           const uint8_t *flags_partitioned, void *out, int64_t *n_out, void *stream) {
    if (!c || !n_out || n < 0 || n != route_n) return fail(c, SPL_E_STATE, "%s", what);
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0) return SPL_OK;
    CK(c, c->rtmp.ensure((size_t)n + 8, 0, st));
    scatter_flags_kernel<<<nblk(n), TILE, 0, st>>>(flags_partitioned, perm, n, c->rtmp.as<uint8_t>());
    const unsigned nt = nblk(n, TILE * 8);
    CKS(c, zero_ctr(c, st));
    CKS(c, prep_status(c, 0, nt, st));
    compact_rows_kernel<<<nt, TILE, 0, st>>>(reinterpret_cast<const R *>(cand), c->rtmp.as<uint8_t>(), n, reinterpret_cast<R *>(out),
                                             c->status[0].as<uint64_t>(), c->d_ctr, 0);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    *n_out = (int64_t)c->h_ctr->n_emitted;
    return SPL_OK;
}

// out[i] = rows[idx[i]] (scatter = 0) or out[idx[i]] = rows[i] (scatter = 1), rows of type R; `fn` names the entry point
template <typename R>
static int move_rows(spl_ctx *c, const char *fn, const void *rows, const int64_t *idx, int64_t n, void *out, int32_t scatter,
                     void *stream) {
    if (!c || n < 0 || (n && (!rows || !idx || !out))) return fail(c, SPL_E_INVALID, "%s: bad arguments", fn);
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    move_rows_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const R *>(rows), idx, n, reinterpret_cast<R *>(out), scatter);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

// ------------------------------------------------------------------ expand + dedup of a level, by kind
// Key-table level: chunks of parents, each expanded straight into probes of the key table, then the winners resolved
// in arrival order into s->uniq (with on-device scores into c->sk).
static int keytable_expand(spl_solver *s, int64_t n, LevelExpand *x, float ms[6], cudaStream_t st) {
    spl_ctx *c = s->c;
    const Rec *front = s->front.as<Rec>();
    int64_t n_uniq = 0, generated = 0;
    uint64_t sk_min = ~0ull, sk_max = 0;
    for (int64_t p0 = 0; p0 < n; p0 += (int64_t)c->chunk_parents) {
        const int64_t np = std::min<int64_t>((int64_t)c->chunk_parents, n - p0);
        const unsigned nt = nblk(np);
        CKS(c, zero_ctr(c, st));
        CK(c, cudaEventRecord(c->ev[0], st));
        CKS(c, run_count(c, front + p0, np, st));
        CK(c, cudaEventRecord(c->ev[7], st));
        const uint64_t total = c->h_ctr->total_cands;
        generated += (int64_t)total;
        if (total == 0) continue;
        if (total >= 0xFFFFFFFFull) return fail(c, SPL_E_INVALID, "chunk produced %llu candidates (>= 2^32)", (unsigned long long)total);
        CKS(c, c->key.grow(c, total, st));
        uint64_t tag;
        CKS(c, next_epoch(c, tag));
        CK(c, c->cand_slot.ensure((size_t)total * 4, 0, st));
        CK(c, cudaEventRecord(c->ev[7], st));
        if (c->identity == IDENT_PYHASH)
            expand_kernel<MODE_PROBE, IDENT_PYHASH><<<nt, TILE, sizeof(ExpandSmem2), st>>>(
                front + p0, np, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(), (uint32_t)total,
                c->key.as<uint64_t>(), c->key.units, tag, c->cand_slot.as<uint32_t>(), nullptr, p0, c->d_ctr);
        else
            expand_kernel<MODE_PROBE, IDENT_KEY><<<nt, TILE, sizeof(ExpandSmem2), st>>>(
                front + p0, np, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(), (uint32_t)total,
                c->key.as<uint64_t>(), c->key.units, tag, c->cand_slot.as<uint32_t>(), nullptr, p0, c->d_ctr);
        ++c->launches;
        CK(c, cudaGetLastError());
        CK(c, cudaEventRecord(c->ev[1], st));
        CKS(c, read_ctr(c, st));
        c->key.occ += c->h_ctr->n_new;  // before the error check: a reset clears a partial insert too
        if (c->h_ctr->error) return fail(c, SPL_E_TABLE_FULL, "visited table full during level %d (slots=%llu, occupied=%llu)",
                                         s->level, (unsigned long long)c->key.slots(), (unsigned long long)c->occupied);
        const int64_t n_new = (int64_t)c->h_ctr->n_new;
        c->occupied += n_new;
        if (n_new) {
            CK(c, s->uniq.ensure((size_t)(n_uniq + n_new) * 32, (size_t)n_uniq * 32, st));
            if (s->use_h) CK(c, c->sk.ensure((size_t)(n_uniq + n_new) * 8, (size_t)n_uniq * 8, st));
            CKS(c, prep_status(c, 0, nt, st));
            CKS(c, reset_ticket(c, 0, st));
            CK(c, cudaEventRecord(c->ev[2], st));
            if (s->use_h && s->noise != SPL_NOISE_EXTERNAL && is_formula_id(s->heuristic))
                resolve_kernel<SRC_PARENT, true, true><<<nt, TILE, sizeof(ResolveSmem), st>>>(
                    front + p0, np, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(), (uint32_t)total,
                    c->key.as<uint64_t>(), c->cand_slot.as<uint32_t>(), nullptr, nullptr, p0, (uint64_t)n_uniq, s->uniq.as<Rec>(),
                    c->sk.as<uint64_t>(), nullptr, s->heuristic, s->noise, c->luts, c->status[0].as<uint64_t>(), c->d_ctr, 0, c->d_forms);
            else if (s->use_h && s->noise != SPL_NOISE_EXTERNAL)
                resolve_kernel<SRC_PARENT, true><<<nt, TILE, sizeof(ResolveSmem), st>>>(
                    front + p0, np, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(), (uint32_t)total,
                    c->key.as<uint64_t>(), c->cand_slot.as<uint32_t>(), nullptr, nullptr, p0, (uint64_t)n_uniq, s->uniq.as<Rec>(),
                    c->sk.as<uint64_t>(), nullptr, s->heuristic, s->noise, c->luts, c->status[0].as<uint64_t>(), c->d_ctr, 0);
            else
                resolve_kernel<SRC_PARENT, false><<<nt, TILE, sizeof(ResolveSmem), st>>>(
                    front + p0, np, c->d_tabs, c->d_takes_idx, c->d_takes_edges, c->off.as<uint32_t>(), (uint32_t)total,
                    c->key.as<uint64_t>(), c->cand_slot.as<uint32_t>(), nullptr, nullptr, p0, (uint64_t)n_uniq, s->uniq.as<Rec>(),
                    nullptr, nullptr, s->heuristic, s->noise, c->luts, c->status[0].as<uint64_t>(), c->d_ctr, 0);
            ++c->launches;
            CK(c, cudaGetLastError());
            CK(c, cudaEventRecord(c->ev[3], st));
            CKS(c, read_ctr(c, st));
            if ((int64_t)c->h_ctr->n_emitted != n_uniq + n_new)
                return fail(c, SPL_E_CUDA, "internal: emitted %llu winners, expected %lld", (unsigned long long)c->h_ctr->n_emitted,
                            (long long)(n_uniq + n_new));
            if (s->use_h && s->noise != SPL_NOISE_EXTERNAL) { sk_min = std::min<uint64_t>(sk_min, c->h_ctr->sk_min); sk_max = std::max<uint64_t>(sk_max, c->h_ctr->sk_max); }
            n_uniq += n_new;
            float t;
            cudaEventElapsedTime(&t, c->ev[2], c->ev[3]);
            ms[2] += t;
        }
        float t;
        cudaEventElapsedTime(&t, c->ev[0], c->ev[7]);
        ms[0] += t;
        cudaEventElapsedTime(&t, c->ev[7], c->ev[1]);
        ms[1] += t;
    }
    *x = LevelExpand{n_uniq, n_uniq, generated, sk_min, sk_max};
    return SPL_OK;
}

// Realistic level: the successors materialised, first-arrival dedup on their exact identity key (src/solver.py:840-843),
// the winners gathered in arrival order into s->uniq.
static int realistic_expand(spl_solver *s, int64_t n, LevelExpand *x, cudaStream_t st) {
    spl_ctx *c = s->c;
    int64_t total = 0, n_new = 0;
    CKS(c, r_expand_all(c, s->front.as<RRec>(), n, 0, &total, st));
    if (total >= 0xFFFFFFFFll) return fail(c, SPL_E_INVALID, "level produced %lld candidates (>= 2^32)", (long long)total);
    if (total) {
        CKS(c, zero_ctr(c, st));
        CKS(c, c->rtab.grow(c, (uint64_t)total, st));
        uint64_t tag;
        CKS(c, next_epoch(c, tag));
        CK(c, c->cand_slot.ensure((size_t)total * 4, 0, st));
        CKS(c, zero_ctr(c, st));
        r_probe_kernel<<<nblk(total), TILE, 0, st>>>(c->rcand.as<RRec>(), total, c->rcfg.as<RConfigDev>(), c->rtab.as<RBucket>(),
                                                      c->rtab.units, tag, c->cand_slot.as<uint32_t>(), c->d_ctr);
        ++c->launches;
        CK(c, cudaGetLastError());
        CKS(c, read_ctr(c, st));
        c->rtab.occ += c->h_ctr->n_new;  // before the error checks: a reset clears a partial insert too
        if (c->h_ctr->error == 4) return fail(c, SPL_E_INVALID, "a player saved 1024 gems or more: outside the packed identity key");
        if (c->h_ctr->error) return fail(c, SPL_E_TABLE_FULL, "visited table full during level %d", s->level);
        n_new = (int64_t)c->h_ctr->n_new;
        c->occupied += n_new;
    }
    if (n_new) {
        CK(c, c->ridx64.ensure((size_t)n_new * 8, 0, st));
        const unsigned nt = nblk(total, TILE * 8);
        CKS(c, prep_status(c, 0, nt, st));
        CKS(c, reset_ticket(c, 0, st));
        r_winners_kernel<<<nt, TILE, 0, st>>>(c->cand_slot.as<uint32_t>(), c->rtab.as<RBucket>(), total, c->ridx64.as<int64_t>(),
                                               c->status[0].as<uint64_t>(), c->d_ctr, 0);
        CK(c, s->uniq.ensure((size_t)n_new * 96, 0, st));
        r_gather_kernel<int64_t><<<nblk(n_new), TILE, 0, st>>>(c->rcand.as<RRec>(), c->ridx64.as<int64_t>(), n_new, s->uniq.as<RRec>());
        c->launches += 2;
        CK(c, cudaGetLastError());
    }
    *x = LevelExpand{n_new, n_new, total, ~0ull, 0};
    return SPL_OK;
}

// ------------------------------------------------------------------ batched levels (spl_rbatch_*, spl_sbatch_*)
// What the two batch kinds share after their expand + dedup: the per-game bookkeeping, the segmented beam cut and the
// end of the level.
//
// Who ends at this level, and the offsets of the winners' runs (useg) and of the next queue's (kseg).  g_host holds per
// game its goal rank (LLONG_MAX: none) | successors | new states.  A game ends when its goal is dequeued, when its queue
// runs out, or at the turn limit (realistic mode: the reference leaves its loop after the iteration with turn == 1000,
// src/solver.py:846-852; the speedrun solver has none).
static int batch_bookkeeping(spl_solver *s, const std::vector<int64_t> &g_host, int64_t n_uniq, bool turn_limit,
                             std::vector<int64_t> &kseg, std::vector<int64_t> &useg, bool *all_ended) {
    RBatch &R = *s->rb;
    const int B = R.B;
    const std::vector<int64_t> &seg = R.seg_at.back();
    kseg.assign(B + 1, 0);
    useg.assign(B + 1, 0);
    *all_ended = true;
    for (int g = 0; g < B; ++g) {
        const int64_t ng = seg[g + 1] - seg[g];
        int64_t kept = 0;
        useg[g + 1] = useg[g];
        if (ng > 0) {
            spl_rgame_info &I = R.info[g];
            const int64_t uniq = (int64_t)g_host[2 * B + g];
            I.level = s->level;
            I.frontier = ng;
            I.goal_rank = -1;
            if (g_host[g] != 0x7fffffffffffffffll) {  // goal dequeued: nothing of this level is expanded
                I.generated = I.unique = I.kept = 0;
                I.goal_rank = R.final_rank[g] = g_host[g];
                I.ended = 1;
            } else {
                I.generated = g_host[B + g];
                I.unique = uniq;
                I.visited += uniq;
                I.kept = std::min(uniq, R.beam[g]);
                if (I.kept == 0 || turn_limit) {  // queue exhausted / turn limit: the last state dequeued ends the game
                    I.ended = 1;
                    R.final_rank[g] = ng - 1;
                } else {
                    kept = I.kept;
                    *all_ended = false;
                }
            }
            useg[g + 1] += uniq;
        }
        kseg[g + 1] = kseg[g] + kept;
    }
    if (useg[B] != n_uniq)
        return fail(s->c, SPL_E_CUDA, "internal: %lld winners, %lld counted per game", (long long)n_uniq, (long long)useg[B]);
    return SPL_OK;
}

// The segmented beam cut: c->y[*cur] / c->idx[*cur] hold the n winners' score sort words (ascending = best first) in a
// stable order, score_bits the low bits in which they differ, rb->uniq_game the winners' games.  One stable sort by
// score, a stable pass by game, then a gather of the first min(beam_g, unique_g) pairs of every game's run into the
// next queue (kseg: its offsets, useg: the winners').  Row: the queue's rows, 96-byte RRec or 32-byte Rec.
template <class Row>
static int segmented_cut(spl_solver *s, int64_t n, int score_bits, const std::vector<int64_t> &kseg, const std::vector<int64_t> &useg,
                         int *cur, cudaStream_t st) {
    spl_ctx *c = s->c;
    RBatch &R = *s->rb;
    const int B = R.B;
    CKS(c, sort_pairs(c, n, score_bits, cur, st));
    if (B > 1) {
        rb_game_words_kernel<<<nblk(n), TILE, 0, st>>>(c->idx[*cur].as<uint32_t>(), R.uniq_game.as<uint32_t>(), n,
                                                        c->y[*cur].as<uint64_t>());
        ++c->launches;
        CKS(c, sort_pairs(c, n, bitlen((uint64_t)B - 1), cur, st));
    }
    std::vector<int64_t> segs(kseg);  // the next queue's offsets, then the winners'
    segs.insert(segs.end(), useg.begin(), useg.end());
    CK(c, cudaMemcpyAsync(R.seg.p, segs.data(), segs.size() * 8, cudaMemcpyHostToDevice, st));
    c->h2d_bytes += segs.size() * 8;
    CK(c, s->front.ensure((size_t)kseg[B] * sizeof(Row), 0, st));
    const int64_t *useg_dev = R.seg.as<int64_t>() + (B + 1), *kseg_dev = R.seg.as<int64_t>();
    if constexpr (std::is_same_v<Row, RRec>)
        rb_cut_kernel<<<nblk(n), TILE, 0, st>>>(s->uniq.as<RRec>(), R.uniq_game.as<uint32_t>(), c->idx[*cur].as<uint32_t>(), n,
                                                 useg_dev, kseg_dev, s->front.as<RRec>());
    else
        sb_cut_kernel<<<nblk(n), TILE, 0, st>>>(s->uniq.as<Rec>(), R.uniq_game.as<uint32_t>(), c->idx[*cur].as<uint32_t>(), n,
                                                 useg_dev, kseg_dev, s->front.as<Rec>());
    ++c->launches;
    CK(c, cudaGetLastError());
    CK(c, cudaStreamSynchronize(st));  // segs is a local
    return SPL_OK;
}

// The end of a batch level: the phase times (events 0..5: count | expand | resolve | select | sort), the aggregate
// counters, and either the end of the batch or the next queue's offsets and link column.
static int batch_finish(spl_solver *s, spl_level_info *info, int64_t n, int64_t total, int64_t n_uniq, const std::vector<int64_t> &kseg,
                        bool all_ended, const VisitTable &table, bool realistic, cudaStream_t st) {
    spl_ctx *c = s->c;
    RBatch &R = *s->rb;
    const int B = R.B;
    const std::vector<int64_t> &seg = R.seg_at.back();
    CK(c, cudaEventRecord(c->ev[5], st));
    CK(c, cudaEventSynchronize(c->ev[5]));
    float t;
    cudaEventElapsedTime(&t, c->ev[0], c->ev[1]); info->ms_count = t;
    cudaEventElapsedTime(&t, c->ev[1], c->ev[2]); info->ms_expand = t;
    cudaEventElapsedTime(&t, c->ev[2], c->ev[3]); info->ms_resolve = t;
    cudaEventElapsedTime(&t, c->ev[3], c->ev[4]); info->ms_select = t;
    cudaEventElapsedTime(&t, c->ev[4], c->ev[5]); info->ms_sort = t;
    info->expanded = n;
    info->generated = total;
    info->unique = n_uniq;
    for (int g = 0; g < B; ++g)
        if (seg[g + 1] > seg[g]) info->kept += R.info[g].kept;
    info->visited = (int64_t)c->occupied;
    info->table_slots = table.slots();
    if (all_ended) {
        s->ended = true;
        info->ended = 1;
        return SPL_OK;
    }
    s->n_front = kseg[B];
    s->level += 1;
    R.seg_at.push_back(kseg);
    CKS(c, save_links(s, s->n_front, realistic, false, st));
    CK(c, cudaStreamSynchronize(st));
    return SPL_OK;
}

// ------------------------------------------------------------------ batched realistic level (spl_rbatch_*)
// One level of every game still running, a fixed sequence of launches whatever the number of games: goal test + count
// (per-game goal ranks and successor counts), expand, probe of (game, key), winners in arrival order, score, then the
// segmented beam cut -- a stable sort of the winners by score, a stable pass by game, and a gather of the first
// min(beam_g, unique_g) pairs of every game's run into the next queue.  The host reads the per-game counters twice
// (after the count and after the probe) and uploads the next queue's offsets once.
static int rbatch_step(spl_solver *s, spl_level_info *info, cudaStream_t st) {
    spl_ctx *c = s->c;
    RBatch &R = *s->rb;
    const int B = R.B;
    const int64_t n = s->n_front;
    long long *goal = R.gctr.as<long long>();
    unsigned long long *cands = R.gctr.as<unsigned long long>() + B, *n_new_g = cands + B;
    std::vector<int64_t> g_host(3 * (size_t)B, 0);  // goal | cands | n_new per game
    for (int g = 0; g < B; ++g) g_host[g] = 0x7fffffffffffffffll;
    // ---- goal test + successor count
    CK(c, cudaEventRecord(c->ev[0], st));
    CK(c, cudaMemcpyAsync(R.gctr.p, g_host.data(), g_host.size() * 8, cudaMemcpyHostToDevice, st));
    CKS(c, zero_ctr(c, st));
    const unsigned nt = nblk(n);
    CK(c, c->off.ensure((size_t)n * 4 + 4, 0, st));
    CK(c, c->rvmask.ensure((size_t)n * 4 + 4, 0, st));
    CKS(c, prep_status(c, 0, nt, st));
    const RConfigDev *cfg = R.cfg.as<RConfigDev>();
    const int64_t *dseg = R.seg.as<int64_t>();
    rb_goal_kernel<<<nt, TILE, 0, st>>>(s->front.as<RRec>(), n, dseg, B, cfg, goal);
    rb_count_scan_kernel<<<nt, TILE, 0, st>>>(s->front.as<RRec>(), n, dseg, B, cfg, goal, c->off.as<uint32_t>(), c->rvmask.as<uint32_t>(),
                                               c->status[0].as<uint64_t>(), c->d_ctr, 0, cands);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(g_host.data(), R.gctr.p, (size_t)B * 16, cudaMemcpyDeviceToHost, st));
    CKS(c, read_ctr(c, st));
    c->d2h_bytes += B * 16;
    CK(c, cudaEventRecord(c->ev[1], st));
    const int64_t total = (int64_t)c->h_ctr->total_cands;
    if (total >= 0xFFFFFFFFll) return fail(c, SPL_E_INVALID, "batch level produced %lld candidates (>= 2^32)", (long long)total);
    // ---- expand + (game, key) dedup + winners in arrival order
    int64_t n_uniq = 0;
    if (total) {
        CK(c, c->rcand.ensure((size_t)total * 96, 0, st));
        CK(c, R.cand_game.ensure((size_t)total * 4, 0, st));
        rb_expand_kernel<<<nt, TILE, 0, st>>>(s->front.as<RRec>(), n, dseg, B, cfg, c->off.as<uint32_t>(), c->rvmask.as<uint32_t>(),
                                               c->rcand.as<RRec>(), R.cand_game.as<uint32_t>());
        ++c->launches;
        CK(c, cudaGetLastError());
        CK(c, cudaEventRecord(c->ev[2], st));
        CKS(c, zero_ctr(c, st));
        CKS(c, c->rbtab.grow(c, (uint64_t)total, st));
        uint64_t tag;
        CKS(c, next_epoch(c, tag));
        CK(c, c->cand_slot.ensure((size_t)total * 4, 0, st));
        CKS(c, zero_ctr(c, st));
        rb_probe_kernel<<<nblk(total), TILE, 0, st>>>(c->rcand.as<RRec>(), R.cand_game.as<uint32_t>(), total, cfg, c->rbtab.as<RBucket>(),
                                                       c->rbtab.units, tag, c->cand_slot.as<uint32_t>(), c->d_ctr, n_new_g);
        ++c->launches;
        CK(c, cudaGetLastError());
        CK(c, cudaMemcpyAsync(g_host.data() + 2 * B, n_new_g, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
        CKS(c, read_ctr(c, st));
        c->d2h_bytes += B * 8;
        c->rbtab.occ += c->h_ctr->n_new;  // before the error checks: a reset clears a partial insert too
        if (c->h_ctr->error == 4) return fail(c, SPL_E_INVALID, "a player saved 1024 gems or more: outside the packed identity key");
        if (c->h_ctr->error) return fail(c, SPL_E_TABLE_FULL, "batch visited table full during level %d", s->level);
        n_uniq = (int64_t)c->h_ctr->n_new;
        c->occupied += n_uniq;
        if (n_uniq) {
            CK(c, c->ridx64.ensure((size_t)n_uniq * 8, 0, st));
            const unsigned wt = nblk(total, TILE * 8);
            CKS(c, prep_status(c, 0, wt, st));
            CKS(c, reset_ticket(c, 0, st));
            r_winners_kernel<<<wt, TILE, 0, st>>>(c->cand_slot.as<uint32_t>(), c->rbtab.as<RBucket>(), total, c->ridx64.as<int64_t>(),
                                                   c->status[0].as<uint64_t>(), c->d_ctr, 0);
            CK(c, s->uniq.ensure((size_t)n_uniq * 96, 0, st));
            CK(c, R.uniq_game.ensure((size_t)n_uniq * 4, 0, st));
            rb_gather_kernel<<<nblk(n_uniq), TILE, 0, st>>>(c->rcand.as<RRec>(), R.cand_game.as<uint32_t>(), c->ridx64.as<int64_t>(), n_uniq,
                                                             s->uniq.as<RRec>(), R.uniq_game.as<uint32_t>());
            c->launches += 2;
            CK(c, cudaGetLastError());
        }
    } else {
        CK(c, cudaEventRecord(c->ev[2], st));
    }
    CK(c, cudaEventRecord(c->ev[3], st));
    // ---- per-game bookkeeping
    std::vector<int64_t> kseg, useg;
    bool all_ended;
    CKS(c, batch_bookkeeping(s, g_host, n_uniq, s->level >= 1000, kseg, useg, &all_ended));
    // ---- score + segmented cut into the next queue
    if (kseg[B]) {
        for (int b = 0; b < 2; ++b) {
            CK(c, c->y[b].ensure((size_t)n_uniq * 8 + 8, 0, st));
            CK(c, c->idx[b].ensure((size_t)n_uniq * 4 + 4, 0, st));
        }
        CKS(c, zero_ctr(c, st));
        rb_score_kernel<<<nblk(n_uniq), TILE, 0, st>>>(s->uniq.as<RRec>(), R.uniq_game.as<uint32_t>(), n_uniq, cfg, c->luts,
                                                        c->y[0].as<uint64_t>(), c->idx[0].as<uint32_t>(), c->d_ctr);
        ++c->launches;
        CK(c, cudaGetLastError());
        CKS(c, read_ctr(c, st));
        CK(c, cudaEventRecord(c->ev[4], st));
        // every score key lies between sk_min and sk_max, so the y words differ only in the low bits where those two do
        int cur = 0;
        CKS(c, segmented_cut<RRec>(s, n_uniq, bitlen(c->h_ctr->sk_min ^ c->h_ctr->sk_max), kseg, useg, &cur, st));
    } else {
        CK(c, cudaEventRecord(c->ev[4], st));
    }
    return batch_finish(s, info, n, total, n_uniq, kseg, all_ended, c->rbtab, true, st);
}

// ------------------------------------------------------------------ batched speedrun level (spl_sbatch_*, spl_sbatch.cuh)
// rbatch_step's sequence over 32-byte rows: goal test + count, expand, probe of (game, key), winners in arrival order,
// score, then -- for the 'det' policy -- stable passes by the inverted key (larger keys first among equal scores), and
// the segmented cut.  A game of exhaustive BFS scores 0 and keeps all its unique states (its beam is unbounded), so the
// stable passes leave them in arrival order, which is its queue order in State.solve.
static int sbatch_step(spl_solver *s, spl_level_info *info, cudaStream_t st) {
    spl_ctx *c = s->c;
    RBatch &R = *s->rb;
    const int B = R.B;
    const int64_t n = s->n_front;
    long long *goal = R.gctr.as<long long>();
    unsigned long long *cands = R.gctr.as<unsigned long long>() + B, *n_new_g = cands + B;
    std::vector<int64_t> g_host(3 * (size_t)B, 0);  // goal | cands | n_new per game
    for (int g = 0; g < B; ++g) g_host[g] = 0x7fffffffffffffffll;
    // ---- goal test + successor count
    CK(c, cudaEventRecord(c->ev[0], st));
    CK(c, cudaMemcpyAsync(R.gctr.p, g_host.data(), g_host.size() * 8, cudaMemcpyHostToDevice, st));
    CKS(c, zero_ctr(c, st));
    const unsigned nt = nblk(n);
    CK(c, c->off.ensure((size_t)n * 4 + 4, 0, st));
    CKS(c, prep_status(c, 0, nt, st));
    const SGame *gm = R.cfg.as<SGame>();
    const int64_t *dseg = R.seg.as<int64_t>();
    sb_goal_kernel<<<nt, TILE, 0, st>>>(s->front.as<Rec>(), n, dseg, B, gm, goal);
    sb_count_scan_kernel<<<nt, TILE, 0, st>>>(s->front.as<Rec>(), n, dseg, B, goal, c->d_tabs, c->d_takes_idx, c->off.as<uint32_t>(),
                                               c->status[0].as<uint64_t>(), c->d_ctr, 0, cands);
    c->launches += 2;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpyAsync(g_host.data(), R.gctr.p, (size_t)B * 16, cudaMemcpyDeviceToHost, st));
    CKS(c, read_ctr(c, st));
    c->d2h_bytes += B * 16;
    CK(c, cudaEventRecord(c->ev[1], st));
    const int64_t total = (int64_t)c->h_ctr->total_cands;
    if (total >= 0xFFFFFFFFll) return fail(c, SPL_E_INVALID, "batch level produced %lld candidates (>= 2^32)", (long long)total);
    // ---- expand + (game, key) dedup + winners in arrival order
    int64_t n_uniq = 0;
    if (total) {
        CK(c, c->tmp_rec.ensure((size_t)total * 32, 0, st));
        CK(c, R.cand_game.ensure((size_t)total * 4, 0, st));
        sb_expand_kernel<<<nt, TILE, 0, st>>>(s->front.as<Rec>(), n, dseg, B, goal, c->d_tabs, c->d_takes_idx, c->d_takes_edges,
                                               c->off.as<uint32_t>(), c->tmp_rec.as<Rec>(), R.cand_game.as<uint32_t>());
        ++c->launches;
        CK(c, cudaGetLastError());
        CK(c, cudaEventRecord(c->ev[2], st));
        CKS(c, zero_ctr(c, st));
        CKS(c, c->sbtab.grow(c, (uint64_t)total, st));
        uint64_t tag;
        CKS(c, next_epoch(c, tag));
        CK(c, c->cand_slot.ensure((size_t)total * 4, 0, st));
        CKS(c, zero_ctr(c, st));
        sb_probe_kernel<<<nblk(total), TILE, 0, st>>>(c->tmp_rec.as<Rec>(), R.cand_game.as<uint32_t>(), total, c->sbtab.as<SBucket>(),
                                                       c->sbtab.units, tag, c->cand_slot.as<uint32_t>(), c->d_ctr, n_new_g);
        ++c->launches;
        CK(c, cudaGetLastError());
        CK(c, cudaMemcpyAsync(g_host.data() + 2 * B, n_new_g, (size_t)B * 8, cudaMemcpyDeviceToHost, st));
        CKS(c, read_ctr(c, st));
        c->d2h_bytes += B * 8;
        c->sbtab.occ += c->h_ctr->n_new;  // before the error check: a reset clears a partial insert too
        if (c->h_ctr->error) return fail(c, SPL_E_TABLE_FULL, "batch visited table full during level %d", s->level);
        n_uniq = (int64_t)c->h_ctr->n_new;
        c->occupied += n_uniq;
        if (n_uniq) {
            CK(c, c->ridx64.ensure((size_t)n_uniq * 8, 0, st));
            const unsigned wt = nblk(total, TILE * 8);
            CKS(c, prep_status(c, 0, wt, st));
            CKS(c, reset_ticket(c, 0, st));
            sb_winners_kernel<<<wt, TILE, 0, st>>>(c->cand_slot.as<uint32_t>(), c->sbtab.as<SBucket>(), total, c->ridx64.as<int64_t>(),
                                                    c->status[0].as<uint64_t>(), c->d_ctr, 0);
            CK(c, s->uniq.ensure((size_t)n_uniq * 32, 0, st));
            CK(c, R.uniq_game.ensure((size_t)n_uniq * 4, 0, st));
            sb_gather_kernel<<<nblk(n_uniq), TILE, 0, st>>>(c->tmp_rec.as<Rec>(), R.cand_game.as<uint32_t>(), c->ridx64.as<int64_t>(), n_uniq,
                                                             s->uniq.as<Rec>(), R.uniq_game.as<uint32_t>());
            c->launches += 2;
            CK(c, cudaGetLastError());
        }
    } else {
        CK(c, cudaEventRecord(c->ev[2], st));
    }
    CK(c, cudaEventRecord(c->ev[3], st));
    // ---- per-game bookkeeping
    std::vector<int64_t> kseg, useg;
    bool all_ended;
    CKS(c, batch_bookkeeping(s, g_host, n_uniq, false, kseg, useg, &all_ended));
    // ---- score (+ key passes) + segmented cut into the next queue
    if (kseg[B]) {
        const bool by_key = s->tie == SPL_TIE_KEY;
        for (int b = 0; b < 2; ++b) {
            CK(c, c->y[b].ensure((size_t)n_uniq * 8 + 8, 0, st));
            CK(c, c->idx[b].ensure((size_t)n_uniq * 4 + 4, 0, st));
        }
        if (by_key) CK(c, c->sk.ensure((size_t)n_uniq * 8, 0, st));
        CKS(c, zero_ctr(c, st));
        uint64_t *score_words = by_key ? c->sk.as<uint64_t>() : c->y[0].as<uint64_t>();  // by key: the key passes come first
        if (s->form)
            sb_score_kernel<true><<<nblk(n_uniq), TILE, 0, st>>>(s->uniq.as<Rec>(), R.uniq_game.as<uint32_t>(), n_uniq, gm, s->noise,
                                                                  c->luts, score_words, c->idx[0].as<uint32_t>(), c->d_ctr, c->d_forms);
        else
            sb_score_kernel<false><<<nblk(n_uniq), TILE, 0, st>>>(s->uniq.as<Rec>(), R.uniq_game.as<uint32_t>(), n_uniq, gm, s->noise,
                                                                   c->luts, score_words, c->idx[0].as<uint32_t>(), c->d_ctr, nullptr);
        ++c->launches;
        CK(c, cudaGetLastError());
        CKS(c, read_ctr(c, st));
        CK(c, cudaEventRecord(c->ev[4], st));
        // the beam games' score keys lie between sk_min and sk_max (none: a level of BFS games only, every word 0)
        const uint64_t kmin = c->h_ctr->sk_min, kmax = c->h_ctr->sk_max;
        int cur = 0;
        if (by_key && kmin <= kmax) {  // least significant first: ~key.lo, ~key.hi over the bits that vary, then the score words
            const uint64_t *rows = s->uniq.as<uint64_t>();
            const int key_bits[2] = {bitlen(c->h_ctr->key_or[0] ^ c->h_ctr->key_and[0]),
                                     bitlen(c->h_ctr->key_or[1] ^ c->h_ctr->key_and[1])};
            for (int w = 0; w < 2; ++w) {
                if (!key_bits[w]) continue;
                sb_words_kernel<<<nblk(n_uniq), TILE, 0, st>>>(c->idx[cur].as<uint32_t>(), n_uniq, rows + w, 4, ~0ull,
                                                                R.uniq_game.as<uint32_t>(), gm, c->y[cur].as<uint64_t>());
                ++c->launches;
                CKS(c, sort_pairs(c, n_uniq, key_bits[w], &cur, st));
            }
            sb_words_kernel<<<nblk(n_uniq), TILE, 0, st>>>(c->idx[cur].as<uint32_t>(), n_uniq, score_words, 1, 0,
                                                            R.uniq_game.as<uint32_t>(), gm, c->y[cur].as<uint64_t>());
            ++c->launches;
            CK(c, cudaGetLastError());
        }
        CKS(c, segmented_cut<Rec>(s, n_uniq, kmin <= kmax ? bitlen(kmin ^ kmax) : 0, kseg, useg, &cur, st));
    } else {
        CK(c, cudaEventRecord(c->ev[4], st));
    }
    return batch_finish(s, info, n, total, n_uniq, kseg, all_ended, c->sbtab, false, st);
}

// ------------------------------------------------------------------ second half of a level
// Score (realistic level, or externally drawn noise: the key-table level scores as it resolves, the grouped level as it
// deduplicates), beam cut (src/solver.py:452-456, :846) and gather of the queue in rank order, or the plain BFS
// hand-over; then the bookkeeping.
static int level_cut(spl_solver *s, spl_level_info *info, int64_t n, const LevelExpand &x, const uint8_t *draws, cudaStream_t st) {
    spl_ctx *c = s->c;
    const bool realistic = s->kind == REALISTIC;
    // the reference leaves its realistic loop after the iteration with turn == 1000 (src/solver.py:846-852): `puzzle` is
    // the last state dequeued from the queue just expanded, which stays in place, and the path has 1001 states
    const bool turn_limit = realistic && s->level >= 1000;
    int64_t kept = x.n_uniq;
    if (s->use_h && kept > 0) {
        uint64_t sk_min = x.sk_min, sk_max = x.sk_max;
        CK(c, cudaEventRecord(c->ev[2], st));
        if (realistic || draws) {
            CKS(c, zero_ctr(c, st));
            CK(c, c->sk.ensure((size_t)x.n_uniq * 8, 0, st));
            if (realistic)
                r_score_kernel<<<nblk(x.n_uniq), TILE, 0, st>>>(s->uniq.as<RRec>(), x.n_uniq, c->rcfg.as<RConfigDev>(), c->luts,
                                                                 c->sk.as<uint64_t>(), nullptr, c->d_ctr, draws);
            else if (is_formula_id(s->heuristic))
                score_rec_kernel<<<nblk(x.n_uniq), TILE, 0, st>>>(s->uniq.as<Rec>(), draws, x.n_uniq,
                                                                   c->d_forms + (s->heuristic - SPL_H_FORMULA_BASE), SPL_NOISE_EXTERNAL,
                                                                   c->sk.as<uint64_t>(), c->d_ctr);
            else
                score_ext_kernel<<<nblk(x.n_uniq), TILE, 0, st>>>(s->uniq.as<Rec>(), draws, x.n_uniq, s->heuristic, c->luts,
                                                                   c->sk.as<uint64_t>(), c->d_ctr);
            ++c->launches;
            CK(c, cudaGetLastError());
            CKS(c, read_ctr(c, st));
            sk_min = c->h_ctr->sk_min;
            sk_max = c->h_ctr->sk_max;
        }
        CK(c, cudaEventRecord(c->ev[4], st));
        CutMode mode;
        if (s->tie == SPL_TIE_KEY) mode.ties = TIES_KEY;
        else if (s->kind == GROUPED) mode = {TIES_LINK, 8 + bitlen((uint64_t)n)};  // unordered winners: arrival order is in their links
        int which = 0;
        CKS(c, run_cut_sort(c, c->sk.as<uint64_t>(), realistic ? nullptr : s->uniq.as<Rec>(), x.n_slots, s->beam, sk_min, sk_max,
                            mode, &which, &kept, st, x.n_uniq));
        CK(c, cudaEventRecord(c->ev[5], st));
        if (!turn_limit) {
            CK(c, s->front.ensure((size_t)kept * (realistic ? 96 : 32), 0, st));
            if (realistic)
                r_gather_kernel<uint32_t><<<nblk(kept), TILE, 0, st>>>(s->uniq.as<RRec>(), c->idx[which].as<uint32_t>(), kept, s->front.as<RRec>());
            else
                gather_rec_kernel<<<nblk(kept), TILE, 0, st>>>(s->uniq.as<Rec>(), c->idx[which].as<uint32_t>(), kept, s->front.as<Rec>());
            ++c->launches;
        }
        CK(c, cudaGetLastError());
        CK(c, cudaEventRecord(c->ev[6], st));
        CK(c, cudaStreamSynchronize(st));
        float t;
        if (realistic) {
            cudaEventElapsedTime(&t, c->ev[2], c->ev[6]);
            info->ms_select = t;  // score + cut + gather
        } else {
            cudaEventElapsedTime(&t, c->ev[4], c->ev[5]);
            info->ms_select = t;  // select + cut + sort
            cudaEventElapsedTime(&t, c->ev[5], c->ev[6]);
            info->ms_sort = t;    // gather into rank order
        }
    } else if (kept > 0) {
        s->front.swap(s->uniq);
    }
    info->kept = kept;
    info->visited = (int64_t)c->occupied;
    info->table_slots = visited_table(c, s->kind).slots();
    if (kept == 0 || turn_limit) {  // queue exhausted: `puzzle` is the last dequeued state (src/solver.py:438,459);
        s->ended = true;            // s->front still holds the level that was just expanded
        s->goal_rank = n - 1;
        info->ended = 1;
        return SPL_OK;
    }
    s->n_front = kept;
    s->level += 1;
    CKS(c, save_links(s, s->n_front, realistic, false, st));
    CK(c, cudaStreamSynchronize(st));
    return SPL_OK;
}

// The row checks of every speedrun create, on the host before any kernel sees a row: a gem hand without a rank indexes
// past a node's bitmap, and a key bit at or above 105 is outside the card set.  `what` names a row in the message
// ("row" of a queue, "game" of a batch).
static int check_rows(spl_ctx *c, const char *fn, const char *what, const Rec *rows, int64_t n) {
    const HostTables &T = host_tables();
    for (int64_t i = 0; i < n; ++i) {
        if (T.gemrank[rows[i].lo & GEM_MASK] == 0xFFFF)
            return fail(c, SPL_E_INVALID, "%s: %s %lld has an illegal gem hand (0x%llx)", fn, what, (long long)i,
                        (unsigned long long)(rows[i].lo & GEM_MASK));
        if (rows[i].hi & ~HI_KEY_MASK)
            return fail(c, SPL_E_INVALID, "%s: %s %lld has a key bit at or above 105", fn, what, (long long)i);
    }
    return SPL_OK;
}

// The speedrun solver's create from a level-0 queue rows[0..n) (links ~0), checked on the host (check_rows; a second
// row with the same key would be a state registered twice).
static int create_solver(spl_ctx *c, const char *fn, const Rec *rows, int64_t n, int32_t goal, int32_t use_h,
                         int32_t heuristic, int64_t beam, int32_t tie, int32_t noise, int32_t keep_links, spl_solver **out) {
    if (use_h && beam < 1) return fail(c, SPL_E_INVALID, "%s: beam_width must be >= 1", fn);
    if (use_h && tie != SPL_TIE_STABLE && tie != SPL_TIE_KEY) return fail(c, SPL_E_INVALID, "%s: unknown tie policy %d", fn, tie);
    if (noise < 0 || noise > SPL_NOISE_EXTERNAL) return fail(c, SPL_E_INVALID, "%s: unknown noise policy %d", fn, noise);
    CKS(c, check_heuristic(c, fn, heuristic));
    CKS(c, check_rows(c, fn, "row", rows, n));
    if (n > 1) {
        std::vector<int64_t> ord(n);
        for (int64_t i = 0; i < n; ++i) ord[i] = i;
        const auto key_less = [&](int64_t a, int64_t b) { return rows[a].hi != rows[b].hi ? rows[a].hi < rows[b].hi : rows[a].lo < rows[b].lo; };
        std::sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) { return key_less(a, b) || (!key_less(b, a) && a < b); });
        for (int64_t i = 1; i < n; ++i)
            if (!key_less(ord[i - 1], ord[i]))
                return fail(c, SPL_E_INVALID, "%s: row %lld has the same key as row %lld", fn, (long long)ord[i], (long long)ord[i - 1]);
    }
    if (c->active) return fail(c, SPL_E_STATE, "%s: a solver is open on this context (destroy it first)", fn);
    CK(c, enter_device(c));
    spl_solver *s = new spl_solver(c);
    s->goal = goal; s->use_h = use_h; s->heuristic = heuristic; s->beam = beam; s->tie = tie;
    s->noise = noise; s->keep_links = keep_links;
    // beam search with on-device scoring runs on the card-set-grouped level; exhaustive BFS (queue order == arrival
    // order), the reference's hash identity and externally drawn noise (arrival-ordered draws) on the key table
    const bool grouped = use_h && noise != SPL_NOISE_EXTERNAL && c->identity == IDENT_KEY && !getenv("SPL_NO_GROUPED");
    s->kind = grouped ? GROUPED : KEY_TABLE;
    s->n_front = n;
    return open_solver(s, s->kind, rows, n, 32, false, "solver create sync failed", out);
}

extern "C" {

int32_t spl_solver_create(spl_ctx *c, const spl_key *root_key, uint64_t root_aux, int32_t goal, int32_t use_h,
                          int32_t heuristic, int64_t beam, int32_t tie, int32_t noise, int32_t keep_links,
                          spl_solver **out) {
    if (!c || !root_key || !out) return fail(c, SPL_E_INVALID, "spl_solver_create: null argument");
    const Rec r{root_key->lo, root_key->hi & HI_KEY_MASK, root_aux, ~0ull};
    return create_solver(c, "spl_solver_create", &r, 1, goal, use_h, heuristic, beam, tie, noise, keep_links, out);
}

int32_t spl_solver_create_queue(spl_ctx *c, const void *rows_host, int64_t n_rows, int32_t goal, int32_t use_h,
                                int32_t heuristic, int64_t beam, int32_t tie, int32_t noise, int32_t keep_links,
                                spl_solver **out) {
    if (!c || !rows_host || !out || n_rows < 1) return fail(c, SPL_E_INVALID, "spl_solver_create_queue: bad arguments (n_rows >= 1)");
    std::vector<Rec> rows((size_t)n_rows);
    memcpy(rows.data(), rows_host, (size_t)n_rows * sizeof(Rec));
    for (Rec &r : rows) r.link = ~0ull;
    return create_solver(c, "spl_solver_create_queue", rows.data(), n_rows, goal, use_h, heuristic, beam, tie, noise, keep_links, out);
}

int32_t spl_solver_destroy(spl_solver *s) {
    if (s) { cudaSetDevice(s->c->device); cudaDeviceSynchronize(); delete s; }
    return SPL_OK;
}

int32_t spl_solver_step(spl_solver *s, spl_level_info *info, void *stream) {
    if (!s || !info) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    if (s->ended) return fail(c, SPL_E_STATE, "spl_solver_step: the search has already ended");
    if (s->pending) return fail(c, SPL_E_STATE, "spl_solver_step: the previous level still waits for spl_solver_cut");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    memset(info, 0, sizeof *info);
    info->level = s->level;
    info->frontier = s->n_front;
    info->goal_rank = -1;
    if (s->kind == REALISTIC_BATCH) return rbatch_step(s, info, st);
    if (s->kind == SPEEDRUN_BATCH) return sbatch_step(s, info, st);
    const int64_t n = s->n_front;
    const bool realistic = s->kind == REALISTIC;
    if (realistic && c->rcfg_dirty) {  // spl_rscore / spl_rexpand / spl_rmaxpts ran with their own GameConfig in between
        CKS(c, upload_rconfig(c, &s->rcfg, st));
        c->rcfg_dirty = false;
    }
    // ---- goal test on the queue (src/solver.py:443-445; realistic mode: game over on dequeue, :827-829): the first
    // state in queue order that has won ends the search; the states before it would be expanded and discarded.
    CKS(c, zero_ctr(c, st));
    if (realistic) r_goal_kernel<<<nblk(n), TILE, 0, st>>>(s->front.as<RRec>(), n, c->rcfg.as<RConfigDev>(), c->d_ctr);
    else goal_kernel<<<nblk(n), TILE, 0, st>>>(s->front.as<Rec>(), n, s->goal, c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    if (c->h_ctr->goal_rank != 0x7fffffffffffffffll) {
        s->ended = true;
        s->goal_rank = c->h_ctr->goal_rank;
        info->ended = 1;
        info->goal_rank = s->goal_rank;
        info->visited = (int64_t)c->occupied;
        info->table_slots = visited_table(c, s->kind).slots();
        return SPL_OK;
    }
    // ---- expand + dedup
    LevelExpand x;
    float ms[6] = {0, 0, 0, 0, 0, 0};  // count, expand, resolve, select, sort, (grouped level) warp kernel
    if (s->kind == KEY_TABLE) CKS(c, keytable_expand(s, n, &x, ms, st));
    else if (s->kind == GROUPED) CKS(c, grouped_expand(s, n, &x, ms, st));
    else CKS(c, realistic_expand(s, n, &x, st));
    info->expanded = n;
    info->generated = x.generated;
    info->unique = x.n_uniq;
    info->ms_count = ms[0]; info->ms_expand = ms[1]; info->ms_resolve = ms[2]; info->ms_warp = ms[5];
    if (s->use_h && s->noise == SPL_NOISE_EXTERNAL && x.n_uniq > 0) {  // wait for the host's randint draws
        CK(c, cudaStreamSynchronize(st));
        s->pending = true;
        s->pend_n = n;
        s->pend_uniq = x.n_uniq;
        info->kept = -1;
        info->visited = (int64_t)c->occupied;
        info->table_slots = visited_table(c, s->kind).slots();
        s->pend_info = *info;
        return SPL_OK;
    }
    return level_cut(s, info, n, x, nullptr, st);
}

int32_t spl_rexpand(spl_ctx *c, const spl_rconfig *cfg, const void *recs, int64_t n, void *out_recs, int64_t cap,
                    int64_t *n_out, void *stream) {
    if (!c || !n_out || n < 0 || n > (16ll << 20)) return fail(c, SPL_E_INVALID, "spl_rexpand: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0) return SPL_OK;
    CKS(c, upload_rconfig(c, cfg, st));
    int64_t total = 0;
    CKS(c, r_expand_all(c, reinterpret_cast<const RRec *>(recs), n, 0, &total, st));
    *n_out = total;
    if (total > cap) return fail(c, SPL_E_CAPACITY, "spl_rexpand: %lld successors, capacity %lld", (long long)total, (long long)cap);
    if (total) CK(c, cudaMemcpyAsync(out_recs, c->rcand.p, (size_t)total * 96, cudaMemcpyDeviceToDevice, st));
    CK(c, cudaStreamSynchronize(st));
    return SPL_OK;
}

int32_t spl_rscore(spl_ctx *c, const spl_rconfig *cfg, const void *recs, int64_t n, double *scores, void *stream) {
    if (!c || n < 0) return fail(c, SPL_E_INVALID, "spl_rscore: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    CKS(c, upload_rconfig(c, cfg, st));
    r_score_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const RRec *>(recs), n, c->rcfg.as<RConfigDev>(), c->luts,
                                              nullptr, scores, c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_rpack(spl_ctx *c, const spl_rconfig *cfg, const void *recs, int64_t n, uint64_t *keys_out, void *stream) {
    if (!c || n < 0) return fail(c, SPL_E_INVALID, "spl_rpack: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    CKS(c, upload_rconfig(c, cfg, st));
    r_pack_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const RRec *>(recs), n, c->rcfg.as<RConfigDev>(), keys_out);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_rmaxpts(spl_ctx *c, const spl_rconfig *cfg, const void *recs, int64_t n, uint8_t *out, void *stream) {
    if (!c || n < 0) return fail(c, SPL_E_INVALID, "spl_rmaxpts: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    if (n == 0) return SPL_OK;
    CKS(c, upload_rconfig(c, cfg, st));
    r_maxpts_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const RRec *>(recs), n, c->rcfg.as<RConfigDev>(), out);
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_rsolver_create(spl_ctx *c, const spl_rconfig *cfg, const void *root_rec_host, int64_t beam, int32_t keep_links,
                           spl_solver **out) {
    if (!c || !cfg || !root_rec_host || !out) return fail(c, SPL_E_INVALID, "spl_rsolver_create: null argument");
    if (beam < 1) return fail(c, SPL_E_INVALID, "spl_rsolver_create: beam_width must be >= 1");
    NO_LIVE_SOLVER(c, "spl_rsolver_create");
    CK(c, enter_device(c));
    CKS(c, upload_rconfig(c, cfg, 0));
    spl_solver *s = new spl_solver(c);
    s->kind = REALISTIC; s->rcfg = *cfg; s->use_h = 1; s->noise = cfg->noise; s->beam = beam; s->keep_links = keep_links;
    s->goal = cfg->target_points;
    s->n_front = 1;
    c->rcfg_dirty = false;
    return open_solver(s, REALISTIC, root_rec_host, 1, 96, false, "rsolver create sync failed", out);
}

int32_t spl_rsolver_frontier(spl_solver *s, const void **recs, int64_t *n) {
    if (!s || !recs || !n || s->kind != REALISTIC) return SPL_E_INVALID;
    *recs = s->front.p;
    *n = s->n_front;
    return SPL_OK;
}

// ---- batched searches (spl_rbatch_*, spl_sbatch_*)
constexpr int32_t MAX_BATCH_GAMES = 1 << 16;

}  // extern "C"

// What both batch creates share once their arguments are checked: a solver of `kind` with the per-game bookkeeping,
// and on the device the games' configs (cfg_bytes each: RConfigDev or SGame), their roots (row_bytes each), the level-0
// offsets 0 .. B, the per-game counters and the roots' games 0 .. B - 1; then open_solver.
static int open_batch(spl_ctx *c, LevelKind kind, const void *cfgs, size_t cfg_bytes, const void *roots, size_t row_bytes,
                      const int64_t *beams, int32_t n_games, int32_t keep_links, const char *fn, spl_solver **out, int tie = 0,
                      int noise = 0) {
    if (c->active) return fail(c, SPL_E_STATE, "%s: a solver is open on this context (destroy it first)", fn);
    CK(c, enter_device(c));
    spl_solver *s = new spl_solver(c);
    s->kind = kind; s->use_h = 1; s->keep_links = keep_links; s->n_front = n_games; s->tie = tie; s->noise = noise;
    s->rb = std::make_unique<RBatch>();
    RBatch &R = *s->rb;
    R.B = n_games;
    R.beam.assign(beams, beams + n_games);
    R.info.assign((size_t)n_games, spl_rgame_info{});
    for (auto &I : R.info) { I.visited = 1; I.goal_rank = -1; }
    R.final_rank.assign((size_t)n_games, 0);
    std::vector<int64_t> seg((size_t)n_games + 1);
    std::vector<uint32_t> iota((size_t)n_games);
    for (int g = 0; g <= n_games; ++g) seg[g] = g;
    for (int g = 0; g < n_games; ++g) iota[g] = (uint32_t)g;
    R.seg_at.push_back(seg);
    const size_t B = (size_t)n_games;
    const cudaError_t e = [&]() -> cudaError_t {
        cudaError_t r = R.cfg.ensure(B * cfg_bytes, 0, 0);
        if (r == cudaSuccess) r = R.roots.ensure(B * row_bytes, 0, 0);
        if (r == cudaSuccess) r = R.seg.ensure((2 * B + 2) * 8, 0, 0);
        if (r == cudaSuccess) r = R.gctr.ensure(3 * B * 8, 0, 0);
        if (r == cudaSuccess) r = R.cand_game.ensure(B * 4, 0, 0);
        if (r == cudaSuccess) r = cudaMemcpyAsync(R.cfg.p, cfgs, B * cfg_bytes, cudaMemcpyHostToDevice, 0);
        if (r == cudaSuccess) r = cudaMemcpyAsync(R.roots.p, roots, B * row_bytes, cudaMemcpyHostToDevice, 0);
        if (r == cudaSuccess) r = cudaMemcpyAsync(R.seg.p, seg.data(), (B + 1) * 8, cudaMemcpyHostToDevice, 0);
        if (r == cudaSuccess) r = cudaMemsetAsync(R.gctr.p, 0, 3 * B * 8, 0);
        if (r == cudaSuccess) r = cudaMemcpyAsync(R.cand_game.p, iota.data(), B * 4, cudaMemcpyHostToDevice, 0);
        if (r == cudaSuccess) r = cudaStreamSynchronize(0);
        return r;
    }();
    if (e != cudaSuccess) {
        cudaGetLastError();
        delete s;
        return fail(c, e == cudaErrorMemoryAllocation ? SPL_E_NOMEM : SPL_E_CUDA, "%s: %s", fn, cudaGetErrorString(e));
    }
    c->h2d_bytes += B * (cfg_bytes + row_bytes + 8 + 4) + 8;
    return open_solver(s, kind, roots, n_games, row_bytes, false, "batch create sync failed", out);
}

static int batch_games(spl_solver *s, LevelKind kind, const char *fn, spl_rgame_info *out_host, int32_t n_games) {
    if (!s || !out_host || s->kind != kind) return SPL_E_INVALID;
    if (n_games != s->rb->B) return fail(s->c, SPL_E_INVALID, "%s: the batch has %d games", fn, s->rb->B);
    memcpy(out_host, s->rb->info.data(), sizeof(spl_rgame_info) * (size_t)n_games);
    return SPL_OK;
}

static int batch_frontier(spl_solver *s, LevelKind kind, size_t row_bytes, const char *fn, int32_t game, const void **rows_dev,
                          int64_t *n_host) {
    if (!s || !rows_dev || !n_host || s->kind != kind) return SPL_E_INVALID;
    if (game < 0 || game >= s->rb->B) return fail(s->c, SPL_E_INVALID, "%s: no game %d", fn, game);
    const std::vector<int64_t> &seg = s->rb->seg_at.back();
    const bool live = !s->ended;  // the last level's queue was expanded and replaced by nothing
    *rows_dev = static_cast<const char *>(s->front.p) + seg[game] * row_bytes;
    *n_host = live ? seg[game + 1] - seg[game] : 0;
    return SPL_OK;
}

// Walk every game's line back through the link columns, one batched read per level (a spilled column is read where it
// lies, on the host), then rebuild the rows forward from the roots on the device, one thread per game.  Row: RRec
// (rb_line_kernel) or Rec (sb_line_kernel).
template <class Row>
static int batch_lines(spl_solver *s, LevelKind kind, const char *fn, void *rows_host, int64_t cap, int32_t *plies_host) {
    if (!s || !rows_host || !plies_host || s->kind != kind) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    RBatch &R = *s->rb;
    if (!s->ended) return fail(c, SPL_E_STATE, "%s: the batch has not ended", fn);
    if (!s->keep_links) return fail(c, SPL_E_STATE, "%s: solver was created with keep_links = 0", fn);
    CK(c, enter_device(c));
    const int B = R.B;
    int max_plies = 0;
    for (int g = 0; g < B; ++g) {
        plies_host[g] = (int32_t)R.info[g].level;
        max_plies = std::max(max_plies, plies_host[g]);
    }
    if (max_plies + 1 > cap) return fail(c, SPL_E_CAPACITY, "%s: a line needs %d records", fn, max_plies + 1);
    const cudaStream_t st = 0;
    std::vector<int64_t> rank(R.final_rank), at;
    std::vector<int> who;
    std::vector<uint64_t> link;
    std::vector<uint8_t> ords((size_t)B * std::max(max_plies, 1), 0);
    for (int l = max_plies; l >= 1; --l) {
        at.clear();
        who.clear();
        for (int g = 0; g < B; ++g)
            if (plies_host[g] >= l) { who.push_back(g); at.push_back(R.seg_at[l][g] + rank[g]); }
        const int64_t m = (int64_t)at.size();
        link.resize(at.size());
        if (s->links.host[l]) {
            for (int64_t k = 0; k < m; ++k) link[k] = s->links.host[l][at[k]];
        } else {
            CK(c, R.scratch.ensure((size_t)m * 16, 0, st));
            int64_t *d_at = R.scratch.as<int64_t>();
            CK(c, cudaMemcpyAsync(d_at, at.data(), (size_t)m * 8, cudaMemcpyHostToDevice, st));
            rb_pick_kernel<<<nblk(m), TILE, 0, st>>>(s->links.dev[l]->as<uint64_t>(), d_at, m, reinterpret_cast<uint64_t *>(d_at + m));
            ++c->launches;
            CK(c, cudaGetLastError());
            CK(c, cudaMemcpyAsync(link.data(), d_at + m, (size_t)m * 8, cudaMemcpyDeviceToHost, st));
            CK(c, cudaStreamSynchronize(st));
            c->h2d_bytes += m * 8;
            c->d2h_bytes += m * 8;
        }
        for (int64_t k = 0; k < m; ++k) {
            const int g = who[k];
            ords[(size_t)g * max_plies + (l - 1)] = (uint8_t)(link[k] & 0xff);
            rank[g] = (int64_t)(link[k] >> 8);
        }
    }
    const size_t line_recs = (size_t)max_plies + 1;
    CK(c, R.scratch.ensure(ords.size() + (size_t)B * 4 + 16, 0, st));
    CK(c, R.lines.ensure((size_t)B * line_recs * sizeof(Row), 0, st));
    int32_t *d_plies = R.scratch.as<int32_t>();
    uint8_t *d_ords = reinterpret_cast<uint8_t *>(d_plies + B);
    CK(c, cudaMemcpyAsync(d_plies, plies_host, (size_t)B * 4, cudaMemcpyHostToDevice, st));
    CK(c, cudaMemcpyAsync(d_ords, ords.data(), ords.size(), cudaMemcpyHostToDevice, st));
    CKS(c, zero_ctr(c, st));
    if constexpr (std::is_same_v<Row, RRec>)
        rb_line_kernel<<<nblk(B), TILE, 0, st>>>(R.roots.as<RRec>(), R.cfg.as<RConfigDev>(), B, d_plies, d_ords, max_plies,
                                                  R.lines.as<RRec>(), c->d_ctr);
    else
        sb_line_kernel<<<nblk(B), TILE, 0, st>>>(R.roots.as<Rec>(), B, d_plies, d_ords, max_plies, c->d_tabs, c->d_takes_idx,
                                                  c->d_takes_edges, R.lines.as<Rec>(), c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    CK(c, cudaMemcpy2DAsync(rows_host, (size_t)cap * sizeof(Row), R.lines.p, line_recs * sizeof(Row), line_recs * sizeof(Row), (size_t)B,
                            cudaMemcpyDeviceToHost, st));
    CKS(c, read_ctr(c, st));
    c->h2d_bytes += (int64_t)(B * 4 + ords.size());
    c->d2h_bytes += (int64_t)(B * line_recs * sizeof(Row));
    if (c->h_ctr->error) return fail(c, SPL_E_CUDA, "internal: a link ordinal names no successor");
    return SPL_OK;
}

extern "C" {

int32_t spl_rbatch_create(spl_ctx *c, const spl_rconfig *cfgs, const void *root_recs_host, const int64_t *beams, int32_t n_games,
                          int32_t keep_links, spl_solver **out) {
    if (!c || !cfgs || !root_recs_host || !beams || !out) return fail(c, SPL_E_INVALID, "spl_rbatch_create: null argument");
    if (n_games < 1 || n_games > MAX_BATCH_GAMES) return fail(c, SPL_E_INVALID, "spl_rbatch_create: n_games must be 1..%d", MAX_BATCH_GAMES);
    std::vector<RConfigDev> dev((size_t)n_games);
    for (int g = 0; g < n_games; ++g) {
        if (beams[g] < 1) return fail(c, SPL_E_INVALID, "spl_rbatch_create: game %d: beam_width must be >= 1", g);
        if (cfgs[g].noise != SPL_NOISE_CONST && cfgs[g].noise != SPL_NOISE_HASH)
            return fail(c, SPL_E_INVALID, "spl_rbatch_create: game %d: noise must be const or hash (mt draws depend on the other games)", g);
        CKS(c, make_rconfig(c, cfgs + g, dev[g]));
    }
    return open_batch(c, REALISTIC_BATCH, dev.data(), sizeof(RConfigDev), root_recs_host, 96, beams, n_games, keep_links,
                      "spl_rbatch_create", out);
}

int32_t spl_rbatch_games(spl_solver *s, spl_rgame_info *out_host, int32_t n_games) {
    return batch_games(s, REALISTIC_BATCH, "spl_rbatch_games", out_host, n_games);
}

int32_t spl_rbatch_frontier(spl_solver *s, int32_t game, const void **recs_dev, int64_t *n_host) {
    return batch_frontier(s, REALISTIC_BATCH, 96, "spl_rbatch_frontier", game, recs_dev, n_host);
}

int32_t spl_rbatch_lines(spl_solver *s, void *recs_host, int64_t cap, int32_t *plies_host) {
    return batch_lines<RRec>(s, REALISTIC_BATCH, "spl_rbatch_lines", recs_host, cap, plies_host);
}

// ---- batched speedrun search
int32_t spl_sbatch_create(spl_ctx *c, const void *root_rows_host, const int32_t *goals, const int32_t *use_heuristic,
                          const int32_t *heuristics, const int64_t *beams, int32_t n_games, int32_t tie_policy, int32_t noise,
                          int32_t keep_links, spl_solver **out) {
    if (!c || !root_rows_host || !goals || !use_heuristic || !heuristics || !beams || !out)
        return fail(c, SPL_E_INVALID, "spl_sbatch_create: null argument");
    if (n_games < 1 || n_games > MAX_BATCH_GAMES) return fail(c, SPL_E_INVALID, "spl_sbatch_create: n_games must be 1..%d", MAX_BATCH_GAMES);
    if (tie_policy != SPL_TIE_STABLE && tie_policy != SPL_TIE_KEY)
        return fail(c, SPL_E_INVALID, "spl_sbatch_create: tie policy must be stable or key, not %d", tie_policy);
    if (noise != SPL_NOISE_CONST && noise != SPL_NOISE_HASH)
        return fail(c, SPL_E_INVALID, "spl_sbatch_create: noise must be const or hash, not %d (external draws depend on the other games)", noise);
    std::vector<Rec> rows((size_t)n_games);
    memcpy(rows.data(), root_rows_host, rows.size() * sizeof(Rec));
    std::vector<SGame> games((size_t)n_games);
    std::vector<int64_t> beam((size_t)n_games);
    CKS(c, check_rows(c, "spl_sbatch_create", "game", rows.data(), n_games));
    bool form = false;
    for (int g = 0; g < n_games; ++g) {
        if (beams[g] < 1) return fail(c, SPL_E_INVALID, "spl_sbatch_create: game %d: beam_width must be >= 1", g);
        CKS(c, check_heuristic(c, "spl_sbatch_create", heuristics[g]));
        form |= use_heuristic[g] && is_formula_id(heuristics[g]);
        rows[g].link = ~0ull;
        games[g] = SGame{goals[g], use_heuristic[g] ? 1 : 0, heuristics[g], 0};
        beam[g] = use_heuristic[g] ? beams[g] : INT64_MAX;  // BFS keeps every unique state
    }
    CKS(c, open_batch(c, SPEEDRUN_BATCH, games.data(), sizeof(SGame), rows.data(), 32, beam.data(), n_games, keep_links,
                      "spl_sbatch_create", out, tie_policy, noise));
    (*out)->form = form;
    return SPL_OK;
}

int32_t spl_sbatch_games(spl_solver *s, spl_rgame_info *out_host, int32_t n_games) {
    return batch_games(s, SPEEDRUN_BATCH, "spl_sbatch_games", out_host, n_games);
}

int32_t spl_sbatch_frontier(spl_solver *s, int32_t game, const void **rows_dev, int64_t *n_host) {
    return batch_frontier(s, SPEEDRUN_BATCH, 32, "spl_sbatch_frontier", game, rows_dev, n_host);
}

int32_t spl_sbatch_lines(spl_solver *s, void *rows_host, int64_t cap, int32_t *plies_host) {
    return batch_lines<Rec>(s, SPEEDRUN_BATCH, "spl_sbatch_lines", rows_host, cap, plies_host);
}

// ---- realistic mode on the key-sharded driver: rows are 96-byte RRec records (spl_dedup_flags, spl_compact_winners and
// spl_move_rows sit beside their realistic twins)
int32_t spl_rexpand_rows(spl_ctx *c, const spl_rconfig *cfg, const void *front, int64_t n, int64_t rank_base, void *out, int64_t cap,
                         int64_t *n_out, void *stream) {
    if (!c || !cfg || !n_out || n < 0 || n > (16ll << 20) || rank_base < 0) return fail(c, SPL_E_INVALID, "spl_rexpand_rows: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *n_out = 0;
    if (n == 0) return SPL_OK;
    CKS(c, use_rconfig(c, cfg, st));
    int64_t total = 0;
    CKS(c, r_count_scan(c, reinterpret_cast<const RRec *>(front), n, &total, st));
    *n_out = total;
    if (total > cap) return fail(c, SPL_E_CAPACITY, "spl_rexpand_rows: %lld successors, capacity %lld", (long long)total, (long long)cap);
    if (total == 0) return SPL_OK;
    r_expand_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const RRec *>(front), n, c->rcfg.as<RConfigDev>(), c->off.as<uint32_t>(),
                                          c->rvmask.as<uint32_t>(), rank_base, reinterpret_cast<RRec *>(out));
    ++c->launches;
    CK(c, cudaGetLastError());
    return SPL_OK;
}

int32_t spl_rroute_keys(spl_ctx *c, const spl_rconfig *cfg, const void *cand, int64_t n, int32_t n_ranks, uint64_t *send_keys,
                        int64_t *counts_host, void *stream) {
    if (!c || !cfg || !counts_host || n < 0 || n >= (1ll << 32) || n_ranks < 1 || n_ranks > 255 || (n && !send_keys))
        return fail(c, SPL_E_INVALID, "spl_rroute_keys: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    for (int g = 0; g < n_ranks; ++g) counts_host[g] = 0;
    c->rroute_n = -1;
    if (n == 0) { c->rroute_n = 0; return SPL_OK; }
    CKS(c, use_rconfig(c, cfg, st));
    for (int b = 0; b < 2; ++b) {
        CK(c, c->y[b].ensure((size_t)n * 8 + 8, 0, st));
        CK(c, c->idx[b].ensure((size_t)n * 4 + 4, 0, st));
    }
    CK(c, c->rkeys.ensure((size_t)n * RKEY_WORDS * 8, 0, st));
    CK(c, c->rperm.ensure((size_t)n * 4, 0, st));
    CKS(c, zero_ctr(c, st));
    r_route_pack_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const RRec *>(cand), n, c->rcfg.as<RConfigDev>(), (uint32_t)n_ranks,
                                                   c->rkeys.as<uint64_t>(), c->y[0].as<uint64_t>(), c->idx[0].as<uint32_t>(), c->d_ctr);
    ++c->launches;
    const unsigned nt = nblk(n, SORT_TILE);
    const size_t msz = (size_t)SORT_BINS * nt;
    CK(c, c->matrix.ensure(msz * 4, 0, st));
    CK(c, c->matrix2.ensure(msz * 4, 0, st));
    CKS(c, sort_pass(c, 0, 0, c->y[0].as<uint64_t>(), n, 0, nt, msz, st));  // one stable pass: digit = owner
    r_gather_keys_kernel<<<nblk(n), TILE, 0, st>>>(c->rkeys.as<uint64_t>(), c->idx[1].as<uint32_t>(), n, send_keys, c->rperm.as<uint32_t>());
    ++c->launches;
    CK(c, cudaGetLastError());
    std::vector<uint32_t> start;
    CKS(c, read_owner_starts(c, nt, n_ranks + 1, start, st));
    CKS(c, read_ctr(c, st));  // synchronises the reads of the starts too
    if (c->h_ctr->error == 4) return fail(c, SPL_E_INVALID, "a player saved 1024 gems or more: outside the packed identity key");
    owner_counts(start, n_ranks, n, counts_host);
    c->rroute_n = n;
    return SPL_OK;
}

int32_t spl_dedup_flags(spl_ctx *c, const spl_key *keys, int64_t n, uint8_t *flags, void *stream) {
    if (!c || n < 0 || n >= (1ll << 32)) return fail(c, SPL_E_INVALID, "spl_dedup_flags: bad arguments");
    NO_LIVE_SOLVER(c, "spl_dedup_flags");
    return dedup_flags(c, false, keys, n, flags, (cudaStream_t)stream);
}

int32_t spl_rdedup_flags(spl_ctx *c, const uint64_t *keys, int64_t n, uint8_t *flags, void *stream) {
    if (!c || n < 0 || n >= (1ll << 32) || (n && (!keys || !flags))) return fail(c, SPL_E_INVALID, "spl_rdedup_flags: bad arguments");
    NO_LIVE_SOLVER(c, "spl_rdedup_flags");
    return dedup_flags(c, true, keys, n, flags, (cudaStream_t)stream);
}

int32_t spl_compact_winners(spl_ctx *c, const void *cand_rows, int64_t n, const uint8_t *flags_partitioned, void *out_rows,
                            int64_t *n_out, void *stream) {
    return compact_winners<Rec>(c, c ? c->route_n : -1, c ? c->idx[1].as<uint32_t>() : nullptr,
                                "spl_compact_winners: must follow spl_route_keys on the same candidates", cand_rows, n,
                                flags_partitioned, out_rows, n_out, stream);
}

int32_t spl_rcompact_winners(spl_ctx *c, const void *cand, int64_t n, const uint8_t *flags_partitioned, void *out, int64_t *n_out,
                             void *stream) {
    return compact_winners<RRec>(c, c ? c->rroute_n : -1, c ? c->rperm.as<uint32_t>() : nullptr,
                                 "spl_rcompact_winners: must follow spl_rroute_keys on the same candidates", cand, n,
                                 flags_partitioned, out, n_out, stream);
}

int32_t spl_move_rows(spl_ctx *c, const void *rows, const int64_t *idx, int64_t n, void *out_rows, int32_t scatter, void *stream) {
    return move_rows<Rec>(c, "spl_move_rows", rows, idx, n, out_rows, scatter, stream);
}

int32_t spl_rmove_rows(spl_ctx *c, const void *rows, const int64_t *idx, int64_t n, void *out, int32_t scatter, void *stream) {
    return move_rows<RRec>(c, "spl_rmove_rows", rows, idx, n, out, scatter, stream);
}

int32_t spl_rfirst_goal(spl_ctx *c, const spl_rconfig *cfg, const void *front, int64_t n, int64_t *rank_host, void *stream) {
    if (!c || !cfg || !rank_host || n < 0 || (n && !front)) return fail(c, SPL_E_INVALID, "spl_rfirst_goal: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *rank_host = -1;
    if (n == 0) return SPL_OK;
    CKS(c, use_rconfig(c, cfg, st));
    CKS(c, zero_ctr(c, st));
    r_goal_kernel<<<nblk(n), TILE, 0, st>>>(reinterpret_cast<const RRec *>(front), n, c->rcfg.as<RConfigDev>(), c->d_ctr);
    ++c->launches;
    CK(c, cudaGetLastError());
    CKS(c, read_ctr(c, st));
    if (c->h_ctr->goal_rank != 0x7fffffffffffffffll) *rank_host = c->h_ctr->goal_rank;
    return SPL_OK;
}

int32_t spl_rreset_visited(spl_ctx *c, void *stream) {
    if (!c) return SPL_E_INVALID;
    NO_LIVE_SOLVER(c, "spl_rreset_visited");
    cudaStream_t st = (cudaStream_t)stream;
    // the speedrun table is cleared too, as spl_rsolver_create does: both tables share the epoch counter, which can only
    // restart at 0 once neither holds a tag (every spl_rdedup_flags call takes one epoch; TAG_MAX bounds them per search)
    CKS(c, reset_visited(c, st));
    CK(c, c->rtab.clear(st));
    return SPL_OK;
}

int32_t spl_rvisited_count(spl_ctx *c, int64_t *n_host) {
    if (!c || !n_host) return SPL_E_INVALID;
    *n_host = (int64_t)c->rtab.occ;
    return SPL_OK;
}

int32_t spl_solver_cut(spl_solver *s, const uint8_t *draws, int64_t n_draws, spl_level_info *info, void *stream) {
    if (!s || !info) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    if (!s->pending) return fail(c, SPL_E_STATE, "spl_solver_cut: no level is waiting for draws");
    if (!draws || n_draws != s->pend_uniq) return fail(c, SPL_E_INVALID, "spl_solver_cut: need exactly %lld draws", (long long)s->pend_uniq);
    cudaStream_t st = (cudaStream_t)stream;
    CK(c, enter_device(c));
    *info = s->pend_info;
    s->pending = false;
    LevelExpand x;
    x.n_uniq = x.n_slots = s->pend_uniq;
    return level_cut(s, info, s->pend_n, x, draws, st);
}

int32_t spl_solver_frontier(spl_solver *s, const spl_key **keys, const uint64_t **aux, const uint64_t **link, int64_t *n) {
    // AoS view: the three pointers address fields of 32-byte records (stride 32 bytes).
    if (!s || !n) return SPL_E_INVALID;
    const char *b = reinterpret_cast<const char *>(s->front.p);
    if (keys) *keys = reinterpret_cast<const spl_key *>(b);
    if (aux) *aux = reinterpret_cast<const uint64_t *>(b + 16);
    if (link) *link = reinterpret_cast<const uint64_t *>(b + 24);
    *n = s->n_front;
    return SPL_OK;
}

int32_t spl_solver_path(spl_solver *s, int64_t *ranks, int32_t *ordinals, int32_t cap, int32_t *n_moves) {
    if (!s || !ranks || !ordinals || !n_moves) return SPL_E_INVALID;
    spl_ctx *c = s->c;
    if (s->kind == REALISTIC_BATCH) return fail(c, SPL_E_INVALID, "spl_solver_path: a batched solver's lines come from spl_rbatch_lines");
    if (s->kind == SPEEDRUN_BATCH) return fail(c, SPL_E_INVALID, "spl_solver_path: a batched solver's lines come from spl_sbatch_lines");
    if (!s->ended) return fail(c, SPL_E_STATE, "spl_solver_path: the search has not ended");
    if (!s->keep_links) return fail(c, SPL_E_STATE, "spl_solver_path: solver was created with keep_links = 0");
    const int L = s->level;  // level index of the final state
    if (L + 1 > cap) return fail(c, SPL_E_CAPACITY, "spl_solver_path: need %d entries", L + 1);
    CK(c, enter_device(c));
    int64_t r = s->goal_rank;
    for (int l = L; l >= 0; --l) {
        ranks[l] = r;
        if (l > 0) {
            uint64_t link = 0;
            CK(c, s->links.read(l, r, &link));
            if (!s->links.host[l]) c->d2h_bytes += 8;
            ordinals[l - 1] = (int32_t)(link & 0xff);
            r = (int64_t)(link >> 8);
        }
    }
    *n_moves = L;
    return SPL_OK;
}

}  // extern "C"
