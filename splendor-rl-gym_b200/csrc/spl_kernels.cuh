// spl_kernels.cuh -- the sm_100a kernels of the frontier-expansion path.
//
//   count_scan_kernel     per-parent fan-out + exclusive offsets (decoupled look-back)
//   expand_kernel<MODE>   successor enumeration (State.__iter__) fused with the visited-table
//                         probe/insert (MODE_PROBE) or materialising candidates (MODE_LIST)
//   probe_list_kernel     visited-table probe/insert of a materialised candidate list
//   resolve_kernel<SRC>   first-arrival winner resolution + ordered emission (+ scoring)
//   score_kernel          heuristics on a batch
//   sel_* / cut_kernel    radix select of the beam threshold + arrival-order cut
//   sort_* / gather       stable LSD radix sort into rank order
//
// Every kernel is HBM/L2-latency bound integer work: no tensor cores (no dense contraction).
#pragma once
#include "spl_common.cuh"

namespace spl {

struct Counters {            // device-resident scalars, zeroed per use by the host driver
    unsigned long long total_cands;   // candidates in this chunk
    unsigned long long n_new;         // successful inserts in this chunk (== winners)
    unsigned long long n_emitted;     // winners emitted so far in this level
    unsigned long long sk_min, sk_max;  // range of order-preserving score keys in this level
    long long goal_rank;              // min rank with pts >= goal (or LLONG_MAX)
    unsigned int error;               // 1 = probe overflow (table full)
    unsigned int ticket[4];           // dynamic tile tickets
    unsigned long long key_or[2], key_and[2];  // OR / AND of the kept keys (det policy: which key bits vary)
    // card-set-grouped level (spl_m2.cuh): total_cands counts the round's gem takes there
    unsigned long long n_buys;        // buy records of the round
    unsigned int n_runs, n_new_nodes; // equal-hash runs of the round; nodes (card sets) created in the round
    unsigned int n_cls[8];            // runs per candidate-count class (m2_dispatch_kernel)
    unsigned long long n_ties;        // tie_collect_kernel: arrival words collected
};

struct SelState {            // radix-select state (device)
    unsigned long long prefix;  // high bits of the threshold found so far (in x = sk - sk_min space)
    unsigned long long k_rem;   // rank still to resolve inside the current bucket
    unsigned long long c_gt;    // elements strictly above the current bucket
    unsigned long long tie_count;  // size of the bucket chosen by the last pick
    unsigned long long khi, klo;   // det policy: key threshold among score ties (keys >= it are kept)
    unsigned long long rank_t;     // dictionary path: descending rank of the threshold score (~0 = no dictionary)
};

// ------------------------------------------------------------------ per-parent derivation
struct SmemTabs {
    uint64_t buy_lo[NCOL][8];
    uint64_t buy_hi[NCOL][8];
    uint32_t card[SPL_NUM_CARDS + 2];
};

__device__ __forceinline__ void load_tabs(SmemTabs &s, const DevTables *__restrict__ g) {
    const uint64_t *src = reinterpret_cast<const uint64_t *>(g);
    uint64_t *dst = reinterpret_cast<uint64_t *>(&s);
    for (int i = threadIdx.x; i < 2 * NCOL * 8; i += blockDim.x) dst[i] = src[i];
    for (int i = threadIdx.x; i < SPL_NUM_CARDS; i += blockDim.x) s.card[i] = g->card[i];
}

// buys mask (key layout) of one parent: State.__iter__ :360-369
__device__ __forceinline__ void buy_mask(const SmemTabs &s, uint64_t lo, uint64_t hi, uint64_t aux, uint64_t &bm_lo,
                                         uint64_t &bm_hi) {
    const uint32_t g = (uint32_t)(lo & GEM_MASK);
    bm_lo = ~lo;
    bm_hi = ~hi & HI_KEY_MASK;
#pragma unroll
    for (int c = 0; c < NCOL; ++c) {
        uint32_t v = ((g >> (3 * c)) & 7) + (uint32_t)((aux >> (24 + 5 * c)) & 31);
        v = v > 7 ? 7 : v;  // min(g + b, MAX_GEMS)
        bm_lo &= s.buy_lo[c][v];
        bm_hi &= s.buy_hi[c][v];
    }
}
// buys mask and take-table entry of one parent: State.__iter__ :360-369, :381
__device__ __forceinline__ void derive_parent(const SmemTabs &s, const uint32_t *__restrict__ takes_idx, uint64_t lo,
                                              uint64_t hi, uint64_t aux, uint64_t &bm_lo, uint64_t &bm_hi,
                                              uint32_t &nb, uint32_t &tk) {
    buy_mask(s, lo, hi, aux, bm_lo, bm_hi);
    nb = __popcll(bm_lo) + __popcll(bm_hi);
    tk = __ldg(takes_idx + (uint32_t)(lo & GEM_MASK));
}

__device__ __forceinline__ int nth_set_bit64(uint64_t m, int n) {
    const uint32_t l = (uint32_t)m, h = (uint32_t)(m >> 32);
    const int c = __popc(l);
    return n < c ? nth_set_bit32(l, n) : 32 + nth_set_bit32(h, n - c);
}

// ord-th successor of a parent in list(iter(parent)) order: buys ascending, then takes.
// State.buy_card :338-355 / subtract_with_bonus gems.py:116-129 / increase_bonus :141-143
__device__ __forceinline__ void make_child(const SmemTabs &s, const uint16_t *__restrict__ takes_edges, uint64_t lo,
                                           uint64_t hi, uint64_t aux, uint64_t bm_lo, uint64_t bm_hi, uint32_t nb,
                                           uint32_t tk, uint32_t ord, uint64_t &clo, uint64_t &chi, uint64_t &caux) {
    if (ord < nb) {
        const int c0 = __popcll(bm_lo);
        const int pos = (int)ord < c0 ? nth_set_bit64(bm_lo, ord) : 64 + nth_set_bit64(bm_hi, ord - c0);
        const uint32_t cd = s.card[pos - 15];
        const uint32_t g = (uint32_t)(lo & GEM_MASK);
        uint32_t ng = 0, saved = 0;
#pragma unroll
        for (int c = 0; c < NCOL; ++c) {
            const int cost = (cd >> (3 * c)) & 7;
            const int b = (int)((aux >> (24 + 5 * c)) & 31);
            const int gc = (g >> (3 * c)) & 7;
            const int pay = max(cost - b, 0);
            saved += cost - pay;
            ng |= (uint32_t)max(gc - pay, 0) << (3 * c);
        }
        clo = (lo & ~GEM_MASK) | ng;
        chi = hi;
        if (pos < 64) clo |= 1ull << pos; else chi |= 1ull << (pos - 64);
        caux = aux + saved + ((uint64_t)((cd >> 15) & 7) << 16) + (1ull << (24 + 5 * ((cd >> 18) & 7)));
    } else {
        const uint32_t e = __ldg(takes_edges + (tk >> 8) + (ord - nb));
        clo = (lo & ~GEM_MASK) | e;
        chi = hi;
        caux = aux;
    }
}

// ------------------------------------------------------------------ visited table probe
// The table is an array of 64-byte buckets of three slots (one DRAM burst per bucket); buckets are
// probed linearly, slots inside a bucket in order.  A key is inserted into the first empty slot of
// its probe sequence with one 128-bit CAS; slots never become empty again, so every later probe of
// the same key meets that slot before it meets an empty one.
// Returns the slot id (bucket << 2 | slot) the candidate resolved to (new insert, or same-epoch
// duplicate that may still be the first arrival), or DEAD if the key was inserted in an earlier epoch
// or an EARLIER arrival of this epoch already holds the slot.  `tinv` = ~t, t = arrival index in this
// epoch (< 2^32 - 1): atomicMax(~t) keeps the FIRST arrival (src/solver.py:447-450) regardless of
// thread order.  `b` is the home bucket (slot_of(hash_key())).
constexpr uint32_t PROBE_NEXT = 0xFFFFFFFEu;  // slot holds another key: keep probing (not a slot id: slot-in-bucket < 3)
// one slot of bucket B whose key words were read as (a, h) and whose arrival word was read as v
// (v may be stale: it only grows, so "v > tinv" stays true once seen)
__device__ __forceinline__ uint32_t probe_slot(uint64_t *B, uint64_t b, int j, uint64_t a, uint64_t h, uint32_t v,
                                               uint64_t tag, uint64_t klo, uint64_t khi, uint64_t want_hi,
                                               uint32_t tinv32, uint32_t &n_new) {
    unsigned int *tword = reinterpret_cast<unsigned int *>(B + 2) + j;
    const uint32_t id = (uint32_t)(b << 2) | (uint32_t)j;
    bool mine = false;
    if ((a | h) == 0) {  // empty: claim with one 128-bit CAS
        cas128(bucket_key(B, j), 0, 0, klo, want_hi, a, h);
        if ((a | h) == 0) {
            a = klo;
            h = want_hi;
            mine = true;
            ++n_new;
        }
        v = 0;  // a competing claim: its arrival word is ordered by the atomicMax below
    }
    if (a != klo || (h & HI_KEY_MASK) != khi) return PROBE_NEXT;
    if (!mine) {
        if ((h >> TAG_SHIFT) != tag) return DEAD;
        if (v > tinv32) return DEAD;  // an earlier arrival is already registered (~t only grows)
    }
    atomicMax(tword, tinv32);
    return id;
}
// Sector 0 of a bucket = slot 0 and the three arrival words, sector 1 = slots 1 and 2.  At the load
// factors of a search most keys live in slot 0, so most probes read one 32-byte sector, as a plain
// one-slot-per-sector table would, while a full bucket still costs a single DRAM burst.
__device__ __forceinline__ uint32_t probe_at(uint64_t *__restrict__ table, uint64_t nb, uint64_t tag, uint64_t b,
                                             uint64_t klo, uint64_t khi, uint64_t tinv, uint32_t &n_new,
                                             unsigned int *error) {
    const uint64_t want_hi = khi | (tag << TAG_SHIFT);
    const uint32_t tinv32 = (uint32_t)tinv;
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        uint64_t *B = table + (b << 3);
        uint64_t a0, h0, t01, t2, a1, h1, a2, h2;
        ld_u64x4_cg(B, a0, h0, t01, t2);
        uint32_t r = probe_slot(B, b, 0, a0, h0, (uint32_t)t01, tag, klo, khi, want_hi, tinv32, n_new);
        if (r != PROBE_NEXT) return r;
        ld_u64x4_cg(B + 4, a1, h1, a2, h2);
        r = probe_slot(B, b, 1, a1, h1, (uint32_t)(t01 >> 32), tag, klo, khi, want_hi, tinv32, n_new);
        if (r != PROBE_NEXT) return r;
        r = probe_slot(B, b, 2, a2, h2, (uint32_t)t2, tag, klo, khi, want_hi, tinv32, n_new);
        if (r != PROBE_NEXT) return r;
        if (++b == nb) b = 0;
    }
    atomicExch(error, 1u);
    return DEAD;
}
__device__ __forceinline__ uint32_t probe_insert(uint64_t *__restrict__ table, uint64_t nb, uint64_t tag, uint64_t klo,
                                                 uint64_t khi, uint64_t tinv, uint32_t &n_new, unsigned int *error) {
    return probe_at(table, nb, tag, slot_of(hash_key(klo, khi), nb), klo, khi, tinv, n_new, error);
}

// ------------------------------------------------------------------ the reference's own identity (optional)
// State.hash = hash((cards, gems)) (src/solver.py:316; __eq__ compares only this value, :335-336):
// CPython's tuple hash (xxHash-style rounds, Objects/tupleobject.c) over the owned card indices in
// ascending order and the five gem counts; a small int hashes to itself.  With IDENT_PYHASH the
// visited table is keyed by this 64-bit value, so states whose hashes collide merge as they do in
// the reference's dict.  Pinned by tests/golden/pyhash.json.
enum { IDENT_KEY = 0, IDENT_PYHASH = 1 };
__device__ __forceinline__ uint64_t pyh_lane(uint64_t acc, uint64_t lane) {
    acc += lane * 14029467366897019727ull;
    acc = (acc << 31) | (acc >> 33);
    return acc * 11400714785074694791ull;
}
__device__ __forceinline__ uint64_t pyh_finish(uint64_t acc, uint64_t len) {
    acc += len ^ (2870177450012600261ull ^ 3527539ull);
    return acc == ~0ull ? 1546275796ull : acc;
}
__device__ __forceinline__ uint64_t py_state_hash(uint64_t lo, uint64_t hi) {
    uint64_t cards = 2870177450012600261ull, gems = 2870177450012600261ull, n = 0;
    for (uint64_t m = lo >> 15; m; m &= m - 1, ++n) cards = pyh_lane(cards, (uint64_t)(__ffsll((long long)m) - 1));
    for (uint64_t m = hi & HI_KEY_MASK; m; m &= m - 1, ++n) cards = pyh_lane(cards, (uint64_t)(48 + __ffsll((long long)m)));
    cards = pyh_finish(cards, n);
#pragma unroll
    for (int c = 0; c < NCOL; ++c) gems = pyh_lane(gems, (lo >> (3 * c)) & 7);
    gems = pyh_finish(gems, NCOL);
    return pyh_finish(pyh_lane(pyh_lane(2870177450012600261ull, cards), gems), 2);
}
template <int IDENT>
__device__ __forceinline__ uint32_t probe_ident(uint64_t *__restrict__ table, uint64_t cap, uint64_t tag, uint64_t klo,
                                                uint64_t khi, uint64_t tinv, uint32_t &n_new, unsigned int *error) {
    if (IDENT == IDENT_PYHASH) {
        klo = py_state_hash(klo, khi);
        khi = 0;
    }
    return probe_insert(table, cap, tag, klo, khi, tinv, n_new, error);
}
__global__ void __launch_bounds__(TILE) pyhash_kernel(const spl_key *__restrict__ keys, int64_t n,
                                                      uint64_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) out[i] = py_state_hash(keys[i].lo, keys[i].hi & HI_KEY_MASK);
}

// ------------------------------------------------------------------ count + scan
__global__ void __launch_bounds__(TILE) count_scan_kernel(const Rec *__restrict__ front, int64_t n_par,
                                                          const DevTables *__restrict__ tabs,
                                                          const uint32_t *__restrict__ takes_idx,
                                                          uint32_t *__restrict__ off, uint64_t *status,
                                                          Counters *ctr, int ticket_id) {
    __shared__ SmemTabs s;
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    load_tabs(s, tabs);
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t p = (int64_t)tile * TILE + threadIdx.x;
    uint32_t cnt = 0;
    if (p < n_par) {
        Rec r;
        ld_rec(front + p, r);
        uint64_t bl, bh;
        uint32_t nb, tk;
        derive_parent(s, takes_idx, r.lo, r.hi, r.aux, bl, bh, nb, tk);
        cnt = nb + (tk & 0xff);
    }
    uint32_t total;
    const uint32_t excl = block_excl_scan(cnt, warp_sums, total);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, total, 0);
        if (threadIdx.x == 0) {
            s_base = e;
            if ((int64_t)(tile + 1) * TILE >= n_par) ctr->total_cands = e + total;
        }
    }
    __syncthreads();
    if (p < n_par) off[p] = (uint32_t)(s_base + excl);
}

// ------------------------------------------------------------------ expand (+ probe)
enum { MODE_PROBE = 0, MODE_LIST = 1 };

struct ExpandSmem {
    SmemTabs tabs;
    uint64_t lo[TILE], hi[TILE], aux[TILE], bm_lo[TILE], bm_hi[TILE];
    uint32_t tk[TILE], nb[TILE], pref[TILE + 1];
};

// load a tile of parents, derive masks; pref[] = tile-local exclusive candidate offsets
__device__ __forceinline__ void load_tile(ExpandSmem &S, const Rec *__restrict__ front, int64_t n_par,
                                          const uint32_t *__restrict__ takes_idx, const uint32_t *__restrict__ off,
                                          uint32_t total, uint32_t tile, uint32_t &c0, uint32_t &ncand) {
    const int64_t p0 = (int64_t)tile * TILE, p = p0 + threadIdx.x;
    c0 = off[p0];
    const uint32_t c1 = (p0 + TILE < n_par) ? off[p0 + TILE] : total;
    ncand = c1 - c0;
    if (p < n_par) {
        Rec r;
        ld_rec(front + p, r);
        uint64_t bl, bh;
        uint32_t nb, tk;
        derive_parent(S.tabs, takes_idx, r.lo, r.hi, r.aux, bl, bh, nb, tk);
        S.lo[threadIdx.x] = r.lo; S.hi[threadIdx.x] = r.hi; S.aux[threadIdx.x] = r.aux;
        S.bm_lo[threadIdx.x] = bl; S.bm_hi[threadIdx.x] = bh;
        S.tk[threadIdx.x] = tk; S.nb[threadIdx.x] = nb;
        S.pref[threadIdx.x] = off[p] - c0;
    } else {
        S.pref[threadIdx.x] = ncand;
    }
    if (threadIdx.x == 0) S.pref[TILE] = ncand;
}

// parent (tile-local) owning tile-local candidate i
__device__ __forceinline__ uint32_t owner_of(const uint32_t *pref, uint32_t i) {
    uint32_t lo = 0, hi = TILE;
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const uint32_t mid = (lo + hi) >> 1;
        if (pref[mid] <= i) lo = mid; else hi = mid;
    }
    return lo;
}

// gems after buying the card at key bit `pos` (subtract_with_bonus, src/gems.py:116-129); also
// returns the gems saved and the packed card.  The pre-purchase bonus is used (src/solver.py:346-347).
__device__ __forceinline__ uint32_t buy_gems(const SmemTabs &s, uint64_t lo, uint64_t aux, int pos, uint32_t &saved,
                                             uint32_t &cd) {
    cd = s.card[pos - 15];
    const uint32_t g = (uint32_t)(lo & GEM_MASK);
    uint32_t ng = 0;
    saved = 0;
#pragma unroll
    for (int c = 0; c < NCOL; ++c) {
        const int cost = (cd >> (3 * c)) & 7;
        const int b = (int)((aux >> (24 + 5 * c)) & 31);
        const int gc = (g >> (3 * c)) & 7;
        const int pay = max(cost - b, 0);
        saved += cost - pay;
        ng |= (uint32_t)max(gc - pay, 0) << (3 * c);
    }
    return ng;
}
// owns card `pos` (key bit) from now on
__device__ __forceinline__ void set_key_bit(uint64_t &lo, uint64_t &hi, int pos) {
    if (pos < 64) lo |= 1ull << pos; else hi |= 1ull << (pos - 64);
}
// key and aux of the successor that buys card `pos` (State.buy_card :338-355): new gems, the card, saved gems,
// points and bonus
__device__ __forceinline__ void buy_child(const SmemTabs &s, uint64_t lo, uint64_t hi, uint64_t aux, int pos, uint64_t &clo,
                                          uint64_t &chi, uint64_t &caux) {
    uint32_t saved, cd;
    const uint32_t ng = buy_gems(s, lo, aux, pos, saved, cd);
    clo = (lo & ~GEM_MASK) | ng;
    chi = hi;
    set_key_bit(clo, chi, pos);
    caux = aux + saved + ((uint64_t)((cd >> 15) & 7) << 16) + (1ull << (24 + 5 * ((cd >> 18) & 7)));
}
// ordinal of that successor in list(iter(parent)): the buys come first, in ascending card order
__device__ __forceinline__ uint32_t buy_ordinal(uint64_t bm_lo, uint64_t bm_hi, int pos) {
    return pos < 64 ? __popcll(bm_lo & ((1ull << pos) - 1)) : __popcll(bm_lo) + __popcll(bm_hi & ((1ull << (pos - 64)) - 1));
}

constexpr int BUY_WIN = 4096;  // buy-list window (entries) staged in shared memory

struct ExpandSmem2 {
    SmemTabs tabs;
    uint64_t lo[TILE], hi[TILE], aux[TILE];
    uint32_t tk[TILE], nb[TILE], pref[TILE], prefb[TILE + 1];
    uint16_t units[TILE / 32][128];   // per warp: (parent lane << 2 | round) of every 32-take unit
    uint16_t blist[BUY_WIN];          // (parent << 7 | key bit) of every buy successor in the window
    uint32_t warp_sums[TILE / 32 + 1];
};

// One CTA expands one tile of TILE parents.  Successors are enumerated in two divergence-free
// streams -- gem takes (warp-uniform units of 32 consecutive table edges of one parent, coalesced)
// and card buys (a compacted list built by bit iteration) -- and each one probes the visited table
// directly: software lookahead (L2 prefetch / cp.async rings) was measured to lose because the probe
// stream is bound by HBM's random-line service rate (profiles/README.md r1b, r1c).
// Arrival index t = off[parent] + ordinal is unchanged by the processing order.
template <int MODE, int IDENT>
__global__ void __launch_bounds__(TILE) expand_kernel(const Rec *__restrict__ front, int64_t n_par,
                                                      const DevTables *__restrict__ tabs,
                                                      const uint32_t *__restrict__ takes_idx,
                                                      const uint16_t *__restrict__ takes_edges,
                                                      const uint32_t *__restrict__ off, uint32_t total,
                                                      uint64_t *__restrict__ table, uint64_t cap, uint64_t tag,
                                                      uint32_t *__restrict__ cand_slot, Rec *__restrict__ cand_out,
                                                      int64_t rank_base, Counters *ctr) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ExpandSmem2 &S = *reinterpret_cast<ExpandSmem2 *>(smem_raw);
    const unsigned tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    load_tabs(S.tabs, tabs);
    __syncthreads();
    // ---- parents of this tile
    const int64_t p0 = (int64_t)blockIdx.x * TILE, p = p0 + tid;
    const uint32_t c0 = off[p0];
    uint64_t bm_lo = 0, bm_hi = 0;
    uint32_t nb = 0, tk = 0;
    if (p < n_par) {
        Rec r;
        ld_rec(front + p, r);
        derive_parent(S.tabs, takes_idx, r.lo, r.hi, r.aux, bm_lo, bm_hi, nb, tk);
        S.lo[tid] = r.lo; S.hi[tid] = r.hi; S.aux[tid] = r.aux;
        S.pref[tid] = off[p] - c0;
    }
    S.tk[tid] = tk;
    S.nb[tid] = nb;
    uint32_t total_buys;
    const uint32_t prefb = block_excl_scan(nb, S.warp_sums, total_buys);
    S.prefb[tid] = prefb;
    if (tid == 0) S.prefb[TILE] = total_buys;
    // ---- take units of this warp's 32 parents
    const uint32_t nt_mine = tk & 0xff, my_units = (nt_mine + 31) >> 5;
    const uint32_t uoff = warp_incl_scan(my_units) - my_units;
    const uint32_t nu = __shfl_sync(0xffffffffu, uoff + my_units, 31);
    for (uint32_t r = 0; r < my_units; ++r) S.units[w][uoff + r] = (uint16_t)(lane << 2 | r);
    __syncthreads();
    uint32_t n_new = 0;
    // ---- gem takes (src/solver.py:381-388)
    for (uint32_t u = 0; u < nu; ++u) {
        const uint32_t unit = S.units[w][u], j = (w << 5) + (unit >> 2), q = ((unit & 3) << 5) + lane;
        const uint32_t tkj = S.tk[j];
        if (q < (tkj & 0xff)) {
            const uint32_t e = __ldg(takes_edges + (tkj >> 8) + q);
            const uint64_t klo = (S.lo[j] & ~GEM_MASK) | e, khi = S.hi[j];
            const uint32_t tt = c0 + S.pref[j] + S.nb[j] + q;
            if (MODE == MODE_PROBE) {
                cand_slot[tt] = probe_ident<IDENT>(table, cap, tag, klo, khi, ~(uint64_t)tt, n_new, &ctr->error);
            } else {
                Rec r{klo, khi, S.aux[j], ((uint64_t)(rank_base + p0 + j) << 8) | (S.nb[j] + q)};
                st_rec(cand_out + tt, r);
            }
        }
    }
    // ---- card buys (src/solver.py:369-374), window by window
    for (uint32_t w0 = 0; w0 < total_buys; w0 += BUY_WIN) {
        __syncthreads();
        {   // each parent lists its affordable, not-owned cards in ascending index order
            uint32_t q = prefb;
            uint64_t m = bm_lo;
            while (m) {
                const int pos = __ffsll((long long)m) - 1;
                m &= m - 1;
                if (q >= w0 && q < w0 + BUY_WIN) S.blist[q - w0] = (uint16_t)(tid << 7 | pos);
                ++q;
            }
            m = bm_hi;
            while (m) {
                const int pos = 64 + __ffsll((long long)m) - 1;
                m &= m - 1;
                if (q >= w0 && q < w0 + BUY_WIN) S.blist[q - w0] = (uint16_t)(tid << 7 | pos);
                ++q;
            }
        }
        __syncthreads();
        const uint32_t nbw = min((uint32_t)BUY_WIN, total_buys - w0);
        for (uint32_t i = tid; i < nbw; i += TILE) {
            const uint32_t ent = S.blist[i], j = ent >> 7;
            const int pos = ent & 127;
            uint64_t klo, khi, caux;
            buy_child(S.tabs, S.lo[j], S.hi[j], S.aux[j], pos, klo, khi, caux);
            const uint32_t ord = w0 + i - S.prefb[j];
            const uint32_t tt = c0 + S.pref[j] + ord;
            if (MODE == MODE_PROBE) {
                cand_slot[tt] = probe_ident<IDENT>(table, cap, tag, klo, khi, ~(uint64_t)tt, n_new, &ctr->error);
            } else {
                Rec r{klo, khi, caux, ((uint64_t)(rank_base + p0 + j) << 8) | ord};
                st_rec(cand_out + tt, r);
            }
        }
    }
    if (MODE == MODE_PROBE) {
#pragma unroll
        for (int d = 16; d; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
        if (lane == 0 && n_new) atomicAdd(&ctr->n_new, (unsigned long long)n_new);
    }
}

// probe/insert of a materialised candidate list (stage operator spl_dedup; multi-GPU owner side)
template <int IDENT>
__global__ void __launch_bounds__(TILE) probe_list_kernel(const spl_key *__restrict__ keys, int64_t n,
                                                          uint64_t *__restrict__ table, uint64_t cap, uint64_t tag,
                                                          uint32_t *__restrict__ cand_slot, Counters *ctr) {
    const int64_t t = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint32_t n_new = 0;
    if (t < n) {
        uint64_t a, b;
        ld_cg_u64x2(reinterpret_cast<const uint64_t *>(keys + t), a, b);
        cand_slot[t] = probe_ident<IDENT>(table, cap, tag, a, b & HI_KEY_MASK, ~(uint64_t)t, n_new, &ctr->error);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
    if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(&ctr->n_new, (unsigned long long)n_new);
}

// ------------------------------------------------------------------ heuristics
// Bit-exact restatement of src/solver.py:210-286: every pow comes from a host-built LUT
// (libm pow, as CPython's float_pow), every * and + is a separately rounded IEEE double
// (__dmul_rn/__dadd_rn cannot be contracted into FMA).
__device__ __forceinline__ double score_state(int h, int noise_mode, uint64_t lo, uint64_t hi, uint64_t aux,
                                              const ScoreLuts &L, int r_ext = 50) {
    const uint32_t pts = (uint32_t)((aux >> 16) & 0xff), saved = (uint32_t)(aux & 0xffff);
    const uint32_t g = (uint32_t)(lo & GEM_MASK);
    uint32_t sum_g = 0, sum_b = 0, nnz = 0;
#pragma unroll
    for (int c = 0; c < NCOL; ++c) {
        sum_g += (g >> (3 * c)) & 7;
        const uint32_t b = (uint32_t)((aux >> (24 + 5 * c)) & 31);
        sum_b += b;
        nnz += b > 0;
    }
    // noise modes: 0 const (randint -> 50), 1 hash, 2 external (the i-th randint(1, 100) of a host-side stream)
    const int r = noise_mode == 1 ? 1 + (int)(mix64(lo, hi) % 100ull) : noise_mode == 2 ? r_ext : 50;
    const double noise = __dmul_rn((double)r, 0.01);
    const int hh = (h >= 0 && h <= 3) ? h : 0;
    const double P = __ldg(L.pts + hh * 256 + pts);
    const double Sv = __ldg(L.saved + hh * 65536 + saved);
    double acc;
    switch (hh) {
        case 1: {  // balanced :218-249
            const uint32_t ncards = __popcll(lo >> 15) + __popcll(hi & HI_KEY_MASK);
            acc = __dadd_rn(__dmul_rn(P, 100.0), __dmul_rn(Sv, 10.0));
            acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 0 * 512 + sum_g + 2 * sum_b), 5.0));
            acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 1 * 512 + ncards), 3.0));
            acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 2 * 512 + nnz), 2.0));
            break;
        }
        case 2:  // aggressive :252-262
            acc = __dadd_rn(__dmul_rn(P, 200.0), __dmul_rn(Sv, 5.0));
            acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 3 * 512 + sum_b), 2.0));
            break;
        case 3:  // efficiency :265-286
            acc = __dadd_rn(__dmul_rn(P, 50.0), __dmul_rn(Sv, 30.0));
            acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 4 * 512 + sum_b), 20.0));
            acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 5 * 512 + nnz), 10.0));
            break;
        default:  // simple :210-215
            acc = __dmul_rn(Sv, P);
            break;
    }
    return __dadd_rn(acc, noise);
}

__global__ void __launch_bounds__(TILE) score_kernel(const spl_key *__restrict__ keys, const uint64_t *__restrict__ aux,
                                                     int64_t n, int h, int noise_mode, ScoreLuts L,
                                                     double *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) out[i] = score_state(h, noise_mode, keys[i].lo, keys[i].hi & HI_KEY_MASK, aux[i], L);
}

// ------------------------------------------------------------------ resolve + ordered emission
enum { SRC_PARENT = 0, SRC_LIST = 1 };
constexpr int MAX_TILE_WORDS = (TILE * 190 + 31) / 32 + 1;  // win bitmask words of a parent tile

struct ResolveSmem {
    ExpandSmem E;
    uint32_t win[MAX_TILE_WORDS];
    uint32_t wpre[MAX_TILE_WORDS];
    uint32_t warp_sums[TILE / 32 + 1];
    uint32_t tile;
    uint64_t base;
};

// One CTA = one tile of TILE parents (SRC_PARENT) or TILE*32 listed candidates (SRC_LIST).
// Pass 1 finds the winners (table slot still holds ~t of the first arrival); look-back turns the
// per-tile winner counts into global output ranks; pass 2 re-derives each winner from its
// parent (no second gather) and writes it, with its score, in arrival order.
template <int SRC, bool SCORE>
__global__ void __launch_bounds__(TILE) resolve_kernel(const Rec *__restrict__ front, int64_t n_par,
                                                       const DevTables *__restrict__ tabs,
                                                       const uint32_t *__restrict__ takes_idx,
                                                       const uint16_t *__restrict__ takes_edges,
                                                       const uint32_t *__restrict__ off, uint32_t total,
                                                       const uint64_t *__restrict__ table,
                                                       const uint32_t *__restrict__ cand_slot,
                                                       const spl_key *__restrict__ list_keys,
                                                       const uint64_t *__restrict__ list_aux, int64_t rank_base,
                                                       uint64_t out_base, Rec *__restrict__ out,
                                                       uint64_t *__restrict__ out_sk, int64_t *__restrict__ out_src,
                                                       int h, int noise_mode, ScoreLuts L, uint64_t *status,
                                                       Counters *ctr, int ticket_id) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ResolveSmem &S = *reinterpret_cast<ResolveSmem *>(smem_raw);
    if (SRC == SRC_PARENT) load_tabs(S.E.tabs, tabs);
    if (threadIdx.x == 0) S.tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = S.tile;
    uint32_t c0, ncand;
    if (SRC == SRC_PARENT) {
        load_tile(S.E, front, n_par, takes_idx, off, total, tile, c0, ncand);
    } else {
        c0 = tile * (TILE * 32u);
        ncand = min((uint32_t)(TILE * 32), total - c0);
    }
    // ---- pass 1: winner flags (4 independent slot gathers in flight per thread)
    const uint32_t nwords = (ncand + 31) >> 5;
    uint32_t mywins = 0;
    for (uint32_t i0 = 0; i0 < ncand; i0 += 4 * TILE) {
        uint32_t sidx[4], v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t i = i0 + k * TILE + threadIdx.x;
            sidx[k] = i < ncand ? cand_slot[c0 + i] : DEAD;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = sidx[k] != DEAD ? ld_cg_u32(slot_tword(table, sidx[k])) : 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t i = i0 + k * TILE + threadIdx.x;
            const bool win = sidx[k] != DEAD && ~v[k] == c0 + i;
            const uint32_t bal = __ballot_sync(0xffffffffu, win);
            if ((threadIdx.x & 31) == 0 && (i >> 5) < nwords) {
                S.win[i >> 5] = bal;
                mywins += __popc(bal);
            }
        }
    }
    uint32_t tile_wins;
    block_excl_scan(mywins, S.warp_sums, tile_wins);
    if (threadIdx.x < 32) {
        const uint64_t e = out_base + lookback_exclusive(status, tile, tile_wins, 0);
        if (threadIdx.x == 0) {
            S.base = e;
            if ((uint64_t)c0 + ncand >= total) ctr->n_emitted = e + tile_wins;
        }
    }
    // ---- word prefix of winner counts (exclusive), processed TILE words at a time
    uint32_t carry = 0;
    for (uint32_t w0 = 0; w0 < nwords; w0 += TILE) {
        const uint32_t w = w0 + threadIdx.x;
        const uint32_t c = w < nwords ? __popc(S.win[w]) : 0;
        uint32_t tot;
        const uint32_t ex = block_excl_scan(c, S.warp_sums, tot);
        if (w < nwords) S.wpre[w] = carry + ex;
        carry += tot;
    }
    __syncthreads();
    // ---- pass 2: emit winners in arrival order, one thread per winner (consecutive threads write
    // consecutive records): winner q of the tile sits in the last word whose exclusive prefix is <= q
    uint64_t kmin = ~0ull, kmax = 0;
    for (uint32_t q = threadIdx.x; q < tile_wins; q += TILE) {
        uint32_t lo_w = 0, hi_w = nwords;  // invariant: wpre[lo_w] <= q < wpre[hi_w] (wpre[nwords] = tile_wins)
        while (hi_w - lo_w > 1) {
            const uint32_t mid = (lo_w + hi_w) >> 1;
            if (S.wpre[mid] <= q) lo_w = mid; else hi_w = mid;
        }
        const uint32_t i = (lo_w << 5) + (uint32_t)nth_set_bit32(S.win[lo_w], (int)(q - S.wpre[lo_w]));
        const uint64_t pos = S.base + q;
        Rec r;
        if (SRC == SRC_PARENT) {
            const uint32_t j = owner_of(S.E.pref, i);
            const uint32_t ord = i - S.E.pref[j];
            make_child(S.E.tabs, takes_edges, S.E.lo[j], S.E.hi[j], S.E.aux[j], S.E.bm_lo[j], S.E.bm_hi[j],
                       S.E.nb[j], S.E.tk[j], ord, r.lo, r.hi, r.aux);
            r.link = ((uint64_t)(rank_base + (int64_t)tile * TILE + j) << 8) | ord;
        } else {
            const uint64_t t = (uint64_t)c0 + i;
            r.lo = list_keys[t].lo;
            r.hi = list_keys[t].hi & HI_KEY_MASK;
            r.aux = list_aux ? list_aux[t] : 0;
            r.link = t;
            if (out_src) out_src[pos] = (int64_t)t;
        }
        st_rec(out + pos, r);
        if (SCORE) {
            const double sc = score_state(h, noise_mode, r.lo, r.hi, r.aux, L);
            const uint64_t k = flip_f64((uint64_t)__double_as_longlong(sc));
            out_sk[pos] = k;
            kmin = min(kmin, k);
            kmax = max(kmax, k);
        }
    }
    if (SCORE) {
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
            kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
        }
        if ((threadIdx.x & 31) == 0 && kmin <= kmax) {
            atomicMin(&ctr->sk_min, (unsigned long long)kmin);
            atomicMax(&ctr->sk_max, (unsigned long long)kmax);
        }
    }
}

// ------------------------------------------------------------------ goal test (src/solver.py:443-445)
__global__ void __launch_bounds__(TILE) goal_kernel(const Rec *__restrict__ front, int64_t n, int goal, Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    long long r = 0x7fffffffffffffffll;
    if (i < n) {
        const uint64_t aux = front[i].aux;
        if ((int)((aux >> 16) & 0xff) >= goal) r = i;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) r = min(r, __shfl_xor_sync(0xffffffffu, r, d));
    if ((threadIdx.x & 31) == 0 && r != 0x7fffffffffffffffll) atomicMin(&ctr->goal_rank, r);
}

// ------------------------------------------------------------------ radix select (beam threshold)
constexpr int SEL_BITS = 11;
constexpr int SEL_BINS = 1 << SEL_BITS;

// Tie key of element i among equal scores.  link_top == 0: the canonical state key (det policy, larger first).
// link_top > 0: the arrival order carried by the record's link word (= parent rank << 8 | ordinal < 2^link_top),
// mapped to lo = 2^link_top - 1 - link so that "larger first" == "earlier arrival first" (stable policy on
// unordered input, spl_m2.cuh).
__device__ __forceinline__ void load_tie_key(const uint64_t *__restrict__ kb, int ks, int64_t i, int link_top, uint64_t &lo,
                                             uint64_t &hi) {
    if (link_top) { lo = ((1ull << link_top) - 1) - kb[i * ks + 3]; hi = 0; }
    else { lo = kb[i * ks]; hi = kb[i * ks + 1]; }
}

// histogram of digit (x >> shift) & (2^bits - 1) over elements whose higher bits equal the prefix.
// WORD 0: x = sk - sk_min (score).  WORD 1 / 2 (det policy): key.hi / key.lo of the elements whose
// score equals the score threshold (and, for WORD 2, whose key.hi equals the hi threshold).
template <int WORD>
// keys are read as kb[i * ks] (lo) and kb[i * ks + 1] (hi): ks = 4 for 32-byte records, 2 for a plain key array
__global__ void __launch_bounds__(TILE) sel_hist_kernel(const uint64_t *__restrict__ sk, const uint64_t *__restrict__ kb,
                                                        int ks, int64_t n, uint64_t sk_min, int shift, int bits, int first,
                                                        const SelState *st, uint32_t *__restrict__ hist, int link_top = 0) {
    __shared__ uint32_t sh[SEL_BINS];
    for (int i = threadIdx.x; i < SEL_BINS; i += TILE) sh[i] = 0;
    __syncthreads();
    const uint64_t prefix = first ? 0 : (WORD == 0 ? st->prefix : WORD == 1 ? st->khi : st->klo);
    const uint64_t T = (WORD == 0 || WORD == 3) ? 0 : st->prefix, Thi = WORD == 2 ? st->khi : 0;
    const int hs = shift + bits;  // bits above the digit must match the prefix
    const uint32_t dmask = (1u << bits) - 1;
    for (int64_t base = (int64_t)blockIdx.x * TILE; base < n; base += (int64_t)gridDim.x * TILE) {
        const int64_t i = base + threadIdx.x;
        bool match = i < n;
        uint64_t x = 0;
        if (match && WORD == 3) {
            x = kb[i];  // compact list of the tie words of the threshold score (tie_collect_kernel)
            match = first || hs >= 64 || (x >> hs) == (prefix >> hs);
        } else if (match) {
            x = sk[i];
            match = x != 0;  // 0 = unused output slot
            x -= sk_min;
            if (WORD > 0 && match) {
                match = x == T;
                if (match) {
                    uint64_t lo, hi;
                    load_tie_key(kb, ks, i, link_top, lo, hi);
                    if (WORD == 1) x = hi;
                    else { match = hi == Thi; x = lo; }
                }
            }
            match = match && (first || hs >= 64 || (x >> hs) == (prefix >> hs));
        }
        const uint32_t d = (uint32_t)(x >> shift) & dmask;
        const unsigned act = __ballot_sync(0xffffffffu, match);
        if (match) {
            const unsigned peers = __match_any_sync(act, d);
            if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(&sh[d], (uint32_t)__popc(peers));
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SEL_BINS; i += TILE)
        if (sh[i]) atomicAdd(&hist[i], sh[i]);
}

// arrival-order ties (link_top > 0): gather the tie words of the elements whose score equals the threshold into a
// compact list, so that the select passes over them read nothing else
__global__ void __launch_bounds__(TILE) tie_collect_kernel(const uint64_t *__restrict__ sk, const uint64_t *__restrict__ kb, int ks,
                                                           int64_t n, uint64_t sk_min, const SelState *st, int link_top,
                                                           uint64_t *__restrict__ list, Counters *ctr) {
    const uint64_t T = st->prefix;
    const unsigned lane = threadIdx.x & 31;
    for (int64_t base = (int64_t)blockIdx.x * TILE; base < n; base += (int64_t)gridDim.x * TILE) {
        const int64_t i = base + threadIdx.x;
        const uint64_t v = i < n ? sk[i] : 0;
        const bool tie = v != 0 && v - sk_min == T;
        const unsigned m = __ballot_sync(0xffffffffu, tie);
        if (m) {
            unsigned long long at = 0;
            if (lane == (unsigned)(__ffs(m) - 1)) at = atomicAdd(&ctr->n_ties, (unsigned long long)__popc(m));
            at = __shfl_sync(0xffffffffu, at, __ffs(m) - 1);
            if (tie) {
                uint64_t lo, hi;
                load_tie_key(kb, ks, i, link_top, lo, hi);
                list[at + __popc(m & ((1u << lane) - 1))] = lo;
            }
        }
    }
}

// choose the bucket holding the k_rem-th largest element; 1 CTA of 1024 threads, 2 bins each.
// `first` = first pass of this word (its prefix starts at 0); `init_k` = very first pass (k_rem = k).
__global__ void __launch_bounds__(1024) sel_pick_kernel(uint32_t *hist, int word, int shift, int first, int init_k,
                                                        uint64_t k, SelState *st) {
    __shared__ unsigned long long s_scan[1024];
    const int t = threadIdx.x;
    const uint32_t h0 = hist[SEL_BINS - 1 - 2 * t], h1 = hist[SEL_BINS - 2 - 2 * t];  // descending bins
    hist[SEL_BINS - 1 - 2 * t] = 0;
    hist[SEL_BINS - 2 - 2 * t] = 0;
    s_scan[t] = (unsigned long long)h0 + h1;
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        unsigned long long v = t >= d ? s_scan[t - d] : 0;
        __syncthreads();
        s_scan[t] += v;
        __syncthreads();
    }
    unsigned long long *pf = word == 0 ? &st->prefix : word == 1 ? &st->khi : &st->klo;
    const unsigned long long k_rem = init_k ? k : st->k_rem;
    const unsigned long long c_gt = init_k ? 0 : st->c_gt;
    const unsigned long long prefix = first ? 0 : *pf;
    const unsigned long long incl = s_scan[t], excl = incl - ((unsigned long long)h0 + h1);
    __syncthreads();
    if (excl < k_rem && k_rem <= incl) {
        unsigned long long above = excl, cnt = h0;
        int bin = SEL_BINS - 1 - 2 * t;
        if (above + h0 < k_rem) { above += h0; bin -= 1; cnt = h1; }
        *pf = prefix | ((unsigned long long)bin << shift);
        st->k_rem = k_rem - above;
        st->c_gt = c_gt + above;
        st->tie_count = cnt;
    }
}

// ------------------------------------------------------------------ score dictionary (beam threshold, few distinct scores)
// The heuristics map a state to one of a few hundred distinct doubles per level (points, bonuses and
// savings are small integers; noise `const` adds the same draw to every state).  One pass counts the
// distinct scores in a small hash table, a single CTA sorts them, finds the threshold score and its
// tie quota, and numbers the scores by descending rank; the cut then emits that rank instead of the
// 64-bit score, so the rank sort needs ceil(log2(distinct)/8) passes instead of up to 8.  More than
// DICT_MAX distinct scores (noise `hash` / `mt` on large levels): the radix select above is used.
constexpr int DICT_CAP = 1 << 14;    // hash slots
constexpr int DICT_MAX = 2048;       // most distinct scores the dictionary path handles
constexpr int DICT_LOCAL = 1024;     // per-CTA staging slots
constexpr unsigned long long DICT_EMPTY = ~0ull;  // not a score: flip_f64 never yields all ones

struct ScoreDict {
    unsigned long long key[DICT_CAP];  // distinct order-preserving score keys
    unsigned int cnt[DICT_CAP];        // occurrences
    unsigned int rank[DICT_CAP];       // descending rank (dict_rank_kernel)
    unsigned int n, over;              // distinct scores inserted; 1 = too many, dictionary abandoned
};

__device__ __forceinline__ uint32_t dict_hash(unsigned long long v) {
    return (uint32_t)((v * 0x9E3779B97F4A7C15ull) >> 40);
}
__device__ __forceinline__ void dict_add(ScoreDict *d, unsigned long long v, unsigned int c) {
    uint32_t s = dict_hash(v) & (DICT_CAP - 1);
    for (int p = 0; p < DICT_CAP; ++p, s = (s + 1) & (DICT_CAP - 1)) {
        unsigned long long cur = *reinterpret_cast<volatile unsigned long long *>(&d->key[s]);
        if (cur != v) {
            if (cur != DICT_EMPTY) continue;
            if (*reinterpret_cast<volatile unsigned int *>(&d->over)) return;
            cur = atomicCAS(&d->key[s], DICT_EMPTY, v);
            if (cur == DICT_EMPTY) {
                if (atomicAdd(&d->n, 1u) >= (unsigned)DICT_MAX) atomicExch(&d->over, 1u);
            } else if (cur != v) {
                continue;
            }
        }
        atomicAdd(&d->cnt[s], c);
        return;
    }
    atomicExch(&d->over, 1u);
}
__device__ __forceinline__ uint32_t dict_rank_of(const ScoreDict *__restrict__ d, unsigned long long v) {
    uint32_t s = dict_hash(v) & (DICT_CAP - 1);
    for (int p = 0; p < DICT_CAP && __ldg(&d->key[s]) != v; ++p) s = (s + 1) & (DICT_CAP - 1);
    return __ldg(&d->rank[s]);
}

__global__ void __launch_bounds__(TILE) dict_build_kernel(const uint64_t *__restrict__ sk, int64_t n, ScoreDict *d) {
    __shared__ unsigned long long lkey[DICT_LOCAL];
    __shared__ unsigned int lcnt[DICT_LOCAL];
    for (int i = threadIdx.x; i < DICT_LOCAL; i += TILE) { lkey[i] = DICT_EMPTY; lcnt[i] = 0; }
    __syncthreads();
    const unsigned lane = threadIdx.x & 31;
    int iter = 0;
    for (int64_t base = (int64_t)blockIdx.x * TILE; base < n; base += (int64_t)gridDim.x * TILE, ++iter) {
        if ((iter & 15) == 15 &&
            __any_sync(0xffffffffu, *reinterpret_cast<volatile unsigned int *>(&d->over) != 0)) break;
        const int64_t i = base + threadIdx.x;
        const unsigned long long v = i < n ? sk[i] : 0;
        const bool ok = v != 0;  // 0 = "no state" (unused output slot of the grouped level); flip_f64 never yields it
        const unsigned act = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const unsigned peers = __match_any_sync(act, v);
            if (lane == (unsigned)(__ffs(peers) - 1)) {
                const unsigned int c = (unsigned int)__popc(peers);
                uint32_t s = dict_hash(v) & (DICT_LOCAL - 1);
                bool done = false;
                for (int p = 0; p < 16 && !done; ++p, s = (s + 1) & (DICT_LOCAL - 1)) {
                    unsigned long long cur = lkey[s];
                    if (cur != v) {
                        if (cur != DICT_EMPTY) continue;
                        cur = atomicCAS(&lkey[s], DICT_EMPTY, v);
                        if (cur != DICT_EMPTY && cur != v) continue;
                    }
                    atomicAdd(&lcnt[s], c);
                    done = true;
                }
                if (!done) dict_add(d, v, c);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < DICT_LOCAL; i += TILE)
        if (lkey[i] != DICT_EMPTY) dict_add(d, lkey[i], lcnt[i]);
}

// 1 CTA of 1024 threads: sort the distinct scores (descending), locate the k-th largest element,
// publish the threshold in SelState (same fields the radix select leaves) and number the scores.
__global__ void __launch_bounds__(1024) dict_rank_kernel(ScoreDict *d, uint64_t k, uint64_t sk_min, SelState *st) {
    __shared__ unsigned long long skey[DICT_MAX];
    __shared__ unsigned int sslot[DICT_MAX];
    __shared__ unsigned long long s_scan[1024];
    __shared__ unsigned int s_n;
    const int t = threadIdx.x;
    if (d->over || d->n > (unsigned)DICT_MAX) {
        if (t == 0) st->rank_t = ~0ull;
        return;
    }
    if (t == 0) s_n = 0;
    for (int i = t; i < DICT_MAX; i += 1024) { skey[i] = 0; sslot[i] = 0xFFFFFFFFu; }  // pads sort last
    __syncthreads();
    for (int s = t; s < DICT_CAP; s += 1024) {
        const unsigned long long kk = d->key[s];
        if (kk != DICT_EMPTY) {
            const unsigned int j = atomicAdd(&s_n, 1u);
            if (j < (unsigned)DICT_MAX) { skey[j] = kk; sslot[j] = (unsigned int)s; }
        }
    }
    __syncthreads();
    const int D = (int)min(s_n, (unsigned)DICT_MAX);
    for (int size = 2; size <= DICT_MAX; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            const int i = ((t / stride) * 2 * stride) + (t % stride), j = i + stride;
            const bool desc = (i & size) == 0;
            const unsigned long long a = skey[i], b = skey[j];
            if (desc ? a < b : a > b) {
                skey[i] = b; skey[j] = a;
                const unsigned int sa = sslot[i];
                sslot[i] = sslot[j]; sslot[j] = sa;
            }
            __syncthreads();
        }
    const int e0 = 2 * t, e1 = 2 * t + 1;
    const unsigned long long c0 = e0 < D ? d->cnt[sslot[e0]] : 0, c1 = e1 < D ? d->cnt[sslot[e1]] : 0;
    s_scan[t] = c0 + c1;
    __syncthreads();
    for (int dd = 1; dd < 1024; dd <<= 1) {
        const unsigned long long v = t >= dd ? s_scan[t - dd] : 0;
        __syncthreads();
        s_scan[t] += v;
        __syncthreads();
    }
    const unsigned long long incl = s_scan[t], excl = incl - (c0 + c1);
    if (excl < k && k <= incl) {
        unsigned long long above = excl, cnt = c0;
        int j = e0;
        if (above + c0 < k) { above += c0; j = e1; cnt = c1; }
        st->prefix = skey[j] - sk_min;
        st->k_rem = k - above;
        st->c_gt = above;
        st->tie_count = cnt;
        st->rank_t = (unsigned long long)j;
    }
    if (e0 < D) d->rank[sslot[e0]] = (unsigned int)e0;
    if (e1 < D) d->rank[sslot[e1]] = (unsigned int)e1;
}

// ------------------------------------------------------------------ beam cut in arrival order
// keep x > T, plus the first k_rem arrivals with x == T (Python's stable sort keeps equal keys in
// arrival order, src/solver.py:453).  Emits (y = sk_max - sk, src index) pairs for the rank sort.
// status_keep carries the running count of elements ABOVE the threshold, status_tie the running count
// of ties: survivors in total = above + min(ties, quota) (read back by the host from the last tile).
#ifndef SPL_CUT_ITEMS
#define SPL_CUT_ITEMS 32
#endif
constexpr int CUT_ITEMS = SPL_CUT_ITEMS;  // 8192 elements per tile (measured: 16 items per thread is no faster, 8 is slower)
// DICT: y = descending rank of the score among the level's distinct scores (ScoreDict)
template <bool DICT>
__global__ void __launch_bounds__(TILE) cut_kernel(const uint64_t *__restrict__ sk, int64_t n, uint64_t sk_min,
                                                   uint64_t sk_max, int keep_all, const SelState *st,
                                                   const ScoreDict *__restrict__ dict,
                                                   uint64_t *__restrict__ out_y, uint32_t *__restrict__ out_idx,
                                                   uint64_t *status_tie, uint64_t *status_keep, Counters *ctr,
                                                   int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_tie_base, s_keep_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t T = keep_all ? 0 : st->prefix, quota = keep_all ? 0 : st->k_rem;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * CUT_ITEMS;
    uint64_t x[CUT_ITEMS];
    uint32_t cnt = 0;  // elements above the threshold (low half) | ties with it (high half); both <= 32
    if (b0 + CUT_ITEMS <= n) {  // the thread's 256 contiguous bytes as 8 x 32-byte loads (whole sectors)
#pragma unroll
        for (int q = 0; q < CUT_ITEMS; q += 4) ld_u64x4(sk + b0 + q, x[q], x[q + 1], x[q + 2], x[q + 3]);
#pragma unroll
        for (int q = 0; q < CUT_ITEMS; ++q) {
            x[q] -= sk_min;
            cnt += (keep_all || x[q] > T) ? 1u : (x[q] == T ? 0x10000u : 0u);
        }
    } else {
#pragma unroll
        for (int q = 0; q < CUT_ITEMS; ++q) {
            x[q] = (b0 + q < n) ? sk[b0 + q] - sk_min : 0;
            if (b0 + q < n) cnt += (keep_all || x[q] > T) ? 1u : (x[q] == T ? 0x10000u : 0u);
        }
    }
    // One block scan and two independent chains walked by two warps at once: elements above the
    // threshold, and ties.  Ties are kept in arrival order up to `quota`, so the survivors before this
    // thread number above_before + min(ties_before, quota).
    uint32_t tot;
    const uint32_t ex = block_excl_scan(cnt, warp_sums, tot);  // tile totals <= 8192: the halves never carry
    if (threadIdx.x < 32) {
        const uint64_t e = keep_all ? 0 : lookback_exclusive(status_tie, tile, tot >> 16, 0);
        if (threadIdx.x == 0) s_tie_base = e;
    } else if (threadIdx.x < 64) {
        const uint64_t e = lookback_exclusive(status_keep, tile, tot & 0xffffu, 0);
        if (threadIdx.x == 32) s_keep_base = e;
    }
    __syncthreads();
    uint64_t tie_rank = s_tie_base + (ex >> 16);
    uint64_t pos = s_keep_base + (ex & 0xffffu) + min(tie_rank, quota);
#pragma unroll
    for (int q = 0; q < CUT_ITEMS; ++q) {
        bool k = false;
        if (b0 + q < n) {
            if (keep_all || x[q] > T) k = true;
            else if (x[q] == T) { k = tie_rank < quota; ++tie_rank; }
        }
        if (k) {
            out_y[pos] = DICT ? (uint64_t)dict_rank_of(dict, x[q] + sk_min) : (sk_max - sk_min) - x[q];
            out_idx[pos] = (uint32_t)(b0 + q);
            ++pos;
        }
    }
}

// det policy (ties -> larger canonical key first): keep x > T, plus the score ties whose key is >=
// the key threshold found by the WORD 1/2 select passes (or every tie when `all_ties`).  Order of
// emission is irrelevant here (the composite sort below fixes the ranks); also accumulates the
// OR / AND of the kept keys so that sort passes over constant key digits can be skipped.
// link_top > 0: tie key = arrival order (load_tie_key).  pack (needs DICT and link_top): emit ONE sort word
// y = score rank << link_top | link (ascending == better first) instead of (y, ~key.lo, ~key.hi).
template <bool DICT>
__global__ void __launch_bounds__(TILE) cut_det_kernel(const uint64_t *__restrict__ sk, const uint64_t *__restrict__ kb,
                                                       int ks, int64_t n, uint64_t sk_min, uint64_t sk_max, int keep_all,
                                                       int all_ties, const SelState *st,
                                                       const ScoreDict *__restrict__ dict, uint64_t *__restrict__ out_y,
                                                       uint64_t *__restrict__ out_klo, uint64_t *__restrict__ out_khi,
                                                       uint32_t *__restrict__ out_idx, uint64_t *status_keep,
                                                       Counters *ctr, int ticket_id, int link_top = 0, int pack = 0) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_keep_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t T = keep_all ? 0 : st->prefix, Thi = st->khi, Tlo = st->klo;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * CUT_ITEMS;
    uint64_t x[CUT_ITEMS], lo[CUT_ITEMS], hi[CUT_ITEMS];
    uint32_t keepmask = 0, kept = 0;
    uint64_t or_lo = 0, or_hi = 0, and_lo = ~0ull, and_hi = ~0ull;
#pragma unroll
    for (int q = 0; q < CUT_ITEMS; ++q) {
        bool k = false;
        const uint64_t v = b0 + q < n ? sk[b0 + q] : 0;
        if (v != 0) {  // 0 = unused output slot
            x[q] = v - sk_min;
            lo[q] = hi[q] = 0;
            if (keep_all || x[q] >= T) load_tie_key(kb, ks, b0 + q, link_top, lo[q], hi[q]);  // states below the cut: score only
            if (keep_all || x[q] > T) k = true;
            else if (x[q] == T) k = all_ties || hi[q] > Thi || (hi[q] == Thi && lo[q] >= Tlo);
            if (k) { or_lo |= lo[q]; or_hi |= hi[q]; and_lo &= lo[q]; and_hi &= hi[q]; }
        }
        keepmask |= (uint32_t)k << q;
        kept += k;
    }
    uint32_t tot;
    const uint32_t keep_ex = block_excl_scan(kept, warp_sums, tot);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status_keep, tile, tot, 0);
        if (threadIdx.x == 0) s_keep_base = e;
    }
    __syncthreads();
    uint64_t pos = s_keep_base + keep_ex;
#pragma unroll
    for (int q = 0; q < CUT_ITEMS; ++q)
        if (keepmask >> q & 1) {
            const uint64_t y = DICT ? (uint64_t)dict_rank_of(dict, x[q] + sk_min) : (sk_max - sk_min) - x[q];
            if (pack) {
                out_y[pos] = (y << link_top) | (((1ull << link_top) - 1) - lo[q]);
            } else {
                out_y[pos] = y;
                out_klo[pos] = ~lo[q];                 // ascending sort of ~key == descending key
                out_khi[pos] = ~hi[q] & HI_KEY_MASK;
            }
            out_idx[pos] = (uint32_t)(b0 + q);
            ++pos;
        }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        or_lo |= __shfl_xor_sync(0xffffffffu, or_lo, d);
        or_hi |= __shfl_xor_sync(0xffffffffu, or_hi, d);
        and_lo &= __shfl_xor_sync(0xffffffffu, and_lo, d);
        and_hi &= __shfl_xor_sync(0xffffffffu, and_hi, d);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicOr(&ctr->key_or[0], (unsigned long long)or_lo);
        atomicOr(&ctr->key_or[1], (unsigned long long)or_hi);
        atomicAnd(&ctr->key_and[0], (unsigned long long)and_lo);
        atomicAnd(&ctr->key_and[1], (unsigned long long)and_hi);
    }
}

// Arrival-order ties on unordered input with a score dictionary (the beam cut of the grouped level): keep x > T and
// the ties whose tie word is >= the selected threshold; emit ONE sort word y = score rank << link_top | link
// (ascending == better first) and the source index.  16 consecutive scores per thread (four 32-byte loads), link
// words are read for ties and survivors only, one block scan and one look-back chain.
constexpr int CUTP_ITEMS = 16;
__global__ void __launch_bounds__(TILE) cut_pack_kernel(const uint64_t *__restrict__ sk, const uint64_t *__restrict__ kb, int ks,
                                                        int64_t n, uint64_t sk_min, int keep_all, int all_ties,
                                                        const SelState *st, const ScoreDict *__restrict__ dict, int link_top,
                                                        uint64_t *__restrict__ out_y, uint32_t *__restrict__ out_idx,
                                                        uint64_t *status_keep, Counters *ctr, int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_keep_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint64_t T = keep_all ? 0 : st->prefix, Tlo = st->klo, LMAX = (1ull << link_top) - 1;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * CUTP_ITEMS;
    uint64_t v[CUTP_ITEMS];
    if (b0 + CUTP_ITEMS <= n) {
#pragma unroll
        for (int q = 0; q < CUTP_ITEMS; q += 4) ld_u64x4(sk + b0 + q, v[q], v[q + 1], v[q + 2], v[q + 3]);
    } else {
#pragma unroll
        for (int q = 0; q < CUTP_ITEMS; ++q) v[q] = b0 + q < n ? sk[b0 + q] : 0;
    }
    uint32_t keepmask = 0;
    uint64_t link[CUTP_ITEMS];
#pragma unroll
    for (int q = 0; q < CUTP_ITEMS; ++q) {
        link[q] = 0;
        if (v[q] == 0) continue;  // unused slot
        const uint64_t x = v[q] - sk_min;
        if (!(keep_all || x >= T)) continue;
        link[q] = kb[(b0 + q) * ks + 3];
        if (keep_all || x > T || all_ties || LMAX - link[q] >= Tlo) keepmask |= 1u << q;
    }
    uint32_t tot;
    const uint32_t keep_ex = block_excl_scan(__popc(keepmask), warp_sums, tot);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status_keep, tile, tot, 0);
        if (threadIdx.x == 0) s_keep_base = e;
    }
    __syncthreads();
    uint64_t pos = s_keep_base + keep_ex;
#pragma unroll
    for (int q = 0; q < CUTP_ITEMS; ++q)
        if (keepmask >> q & 1) {
            out_y[pos] = ((uint64_t)dict_rank_of(dict, v[q]) << link_top) | link[q];
            out_idx[pos] = (uint32_t)(b0 + q);
            ++pos;
        }
}

// ------------------------------------------------------------------ stable LSD radix sort of (y, idx) pairs
constexpr int SORT_BITS = 8;
constexpr int SORT_BINS = 1 << SORT_BITS;
constexpr int SORT_ITEMS = 16;                    // per thread; one warp owns 512 consecutive elements
constexpr int SORT_TILE = TILE * SORT_ITEMS;      // 4096 elements per CTA

__global__ void __launch_bounds__(TILE) sort_hist_kernel(const uint64_t *__restrict__ y, int64_t n, int shift,
                                                         uint32_t *__restrict__ matrix, uint32_t ntiles) {
    __shared__ uint32_t sh[SORT_BINS];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * SORT_TILE;
    for (int q = 0; q < SORT_ITEMS; ++q) {
        const int64_t i = base + q * TILE + threadIdx.x;
        if (i < n) atomicAdd(&sh[(uint32_t)(y[i] >> shift) & (SORT_BINS - 1)], 1u);
    }
    __syncthreads();
    matrix[(uint64_t)threadIdx.x * ntiles + blockIdx.x] = sh[threadIdx.x];  // digit-major
}

// generic exclusive scan of u32 (decoupled look-back), 256 threads x 8 items
constexpr int SCAN_ITEMS = 8;
__global__ void __launch_bounds__(TILE) scan_u32_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                                                        int64_t n, uint64_t *status, Counters *ctr, int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * SCAN_ITEMS;
    uint32_t v[SCAN_ITEMS], sum = 0;
#pragma unroll
    for (int q = 0; q < SCAN_ITEMS; ++q) {
        v[q] = (b0 + q < n) ? in[b0 + q] : 0;
        sum += v[q];
    }
    uint32_t tot;
    uint32_t ex = block_excl_scan(sum, warp_sums, tot);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, tot, 0);
        if (threadIdx.x == 0) s_base = e;
    }
    __syncthreads();
    uint32_t run = (uint32_t)s_base + ex;
#pragma unroll
    for (int q = 0; q < SCAN_ITEMS; ++q)
        if (b0 + q < n) { out[b0 + q] = run; run += v[q]; }
}

// `dig` = the array the digit is taken from (one of the payload arrays).  WIDE also moves the
// two inverted key words (det policy composite sort).
template <bool WIDE>
__global__ void __launch_bounds__(TILE) sort_scatter_kernel(const uint64_t *__restrict__ dig,
                                                            const uint64_t *__restrict__ y_in,
                                                            const uint32_t *__restrict__ idx_in, int64_t n, int shift,
                                                            const uint32_t *__restrict__ matrix_scanned,
                                                            uint32_t ntiles, uint64_t *__restrict__ y_out,
                                                            uint32_t *__restrict__ idx_out,
                                                            const uint64_t *__restrict__ klo_in,
                                                            const uint64_t *__restrict__ khi_in,
                                                            uint64_t *__restrict__ klo_out,
                                                            uint64_t *__restrict__ khi_out) {
    __shared__ uint32_t whist[TILE / 32][SORT_BINS];
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < (TILE / 32) * SORT_BINS; i += TILE) (&whist[0][0])[i] = 0;
    __syncthreads();
    const int64_t wbase = (int64_t)blockIdx.x * SORT_TILE + (int64_t)w * (32 * SORT_ITEMS);
    uint32_t dd[SORT_ITEMS];
    // pass A: per-warp digit counts over the warp's contiguous 512-element segment
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {
        const int64_t i = wbase + q * 32 + lane;
        const bool ok = i < n;
        dd[q] = ok ? (uint32_t)(dig[i] >> shift) & (SORT_BINS - 1) : 0;
        const uint32_t d = dd[q];
        const unsigned act = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const unsigned peers = __match_any_sync(act, d);
            if (lane == (unsigned)(__ffs(peers) - 1)) whist[w][d] += __popc(peers);
        }
        __syncwarp();
    }
    __syncthreads();
    {  // exclusive over warps, plus the tile's global base for each digit
        const uint32_t d = threadIdx.x;
        uint32_t run = matrix_scanned[(uint64_t)d * ntiles + blockIdx.x];
        for (int ww = 0; ww < TILE / 32; ++ww) {
            const uint32_t c = whist[ww][d];
            whist[ww][d] = run;
            run += c;
        }
    }
    __syncthreads();
    // pass B: stable scatter
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {
        const int64_t i = wbase + q * 32 + lane;
        const bool ok = i < n;
        const uint32_t d = dd[q];
        const unsigned act = __ballot_sync(0xffffffffu, ok);
        if (ok) {
            const unsigned peers = __match_any_sync(act, d);
            const uint32_t rank = __popc(peers & ((1u << lane) - 1));
            const uint32_t pos = whist[w][d] + rank;
            y_out[pos] = y_in[i];
            idx_out[pos] = idx_in[i];
            if (WIDE) { klo_out[pos] = klo_in[i]; khi_out[pos] = khi_in[i]; }
            __syncwarp(peers);
            if (lane == (unsigned)(__ffs(peers) - 1)) whist[w][d] += __popc(peers);
        }
        __syncwarp();
    }
}

// inverted key words of the kept elements in their final order (SPL_TIE_KEY_ORDERED: the sort moved only (y, idx))
__global__ void __launch_bounds__(TILE) key_words_kernel(const uint32_t *__restrict__ idx, int64_t n,
                                                         const uint64_t *__restrict__ kb, int ks,
                                                         uint64_t *__restrict__ klo, uint64_t *__restrict__ khi) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        const uint64_t s = idx[i];
        klo[i] = ~kb[s * ks];
        khi[i] = ~kb[s * ks + 1] & HI_KEY_MASK;
    }
}

// frontier[rank] = uniq[idx[rank]]
__global__ void __launch_bounds__(TILE) gather_rec_kernel(const Rec *__restrict__ src, const uint32_t *__restrict__ idx,
                                                          int64_t n, Rec *__restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        Rec r;
        ld_rec(src + idx[i], r);
        st_rec(dst + i, r);
    }
}

__global__ void __launch_bounds__(TILE) idx_widen_kernel(const uint32_t *__restrict__ idx, int64_t n,
                                                         int64_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) out[i] = idx[i];
}

// pack / unpack between the C-ABI SoA views (keys, aux, link) and AoS records
__global__ void __launch_bounds__(TILE) pack_rec_kernel(const spl_key *__restrict__ keys, const uint64_t *__restrict__ aux,
                                                        int64_t n, Rec *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        Rec r{keys[i].lo, keys[i].hi & HI_KEY_MASK, aux ? aux[i] : 0ull, ~0ull};
        st_rec(out + i, r);
    }
}
__global__ void __launch_bounds__(TILE) unpack_rec_kernel(const Rec *__restrict__ in, int64_t n, spl_key *__restrict__ keys,
                                                          uint64_t *__restrict__ aux, uint64_t *__restrict__ link) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        Rec r;
        ld_rec(in + i, r);
        if (keys) { keys[i].lo = r.lo; keys[i].hi = r.hi; }
        if (aux) aux[i] = r.aux;
        if (link) link[i] = r.link;
    }
}
__global__ void __launch_bounds__(TILE) flip_scores_kernel(const double *__restrict__ sc, int64_t n,
                                                           uint64_t *__restrict__ sk, Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint64_t kmin = ~0ull, kmax = 0;
    if (i < n) {
        const uint64_t k = flip_f64((uint64_t)__double_as_longlong(sc[i]));
        sk[i] = k;
        kmin = kmax = k;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
    }
    if ((threadIdx.x & 31) == 0 && kmin <= kmax) {
        atomicMin(&ctr->sk_min, (unsigned long long)kmin);
        atomicMax(&ctr->sk_max, (unsigned long long)kmax);
    }
}

// ------------------------------------------------------------------ multi-GPU building blocks (SURVEY.md 8e)
// owner rank of a key: a second, independent mix of the key so that ownership and the slot index
// inside the owner's table are uncorrelated
__device__ __host__ __forceinline__ uint32_t owner_of_key(uint64_t lo, uint64_t hi, uint32_t n_ranks) {
    uint64_t x = (lo * 0xC2B2AE3D27D4EB4Full) ^ (hi * 0x165667B19E3779F9ull);
    x ^= x >> 29;
    x *= 0xBF58476D1CE4E5B9ull;
    x ^= x >> 32;
    return (uint32_t)(((x & 0xffffffffull) * n_ranks) >> 32);
}
__global__ void __launch_bounds__(TILE) owner_kernel(const spl_key *__restrict__ keys, int64_t n, uint32_t n_ranks,
                                                     uint64_t *__restrict__ y, uint32_t *__restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        y[i] = owner_of_key(keys[i].lo, keys[i].hi & HI_KEY_MASK, n_ranks);
        idx[i] = (uint32_t)i;
    }
}
__global__ void __launch_bounds__(TILE) owner_rows_kernel(const Rec *__restrict__ rows, int64_t n, uint32_t n_ranks,
                                                          uint64_t *__restrict__ y, uint32_t *__restrict__ idx) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        uint64_t lo, hi;
        ld_cg_u64x2(reinterpret_cast<const uint64_t *>(rows + i), lo, hi);
        y[i] = owner_of_key(lo, hi & HI_KEY_MASK, n_ranks);
        idx[i] = (uint32_t)i;
    }
}
// send buffer: keys of the candidates in (owner, arrival) order
__global__ void __launch_bounds__(TILE) gather_keys_kernel(const Rec *__restrict__ rows, const uint32_t *__restrict__ idx,
                                                           int64_t n, spl_key *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        uint64_t lo, hi;
        ld_cg_u64x2(reinterpret_cast<const uint64_t *>(rows + idx[i]), lo, hi);
        out[i].lo = lo;
        out[i].hi = hi;
    }
}
__global__ void __launch_bounds__(TILE) scatter_flags_kernel(const uint8_t *__restrict__ part, const uint32_t *__restrict__ idx,
                                                             int64_t n, uint8_t *__restrict__ arrival) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) arrival[idx[i]] = part[i];
}

// scores of rows[i] with the i-th externally drawn randint (noise policy `mt`): order-preserving keys + range
__global__ void __launch_bounds__(TILE) score_ext_kernel(const Rec *__restrict__ rows, const uint8_t *__restrict__ draws,
                                                         int64_t n, int h, ScoreLuts L, uint64_t *__restrict__ sk,
                                                         Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint64_t kmin = ~0ull, kmax = 0;
    if (i < n) {
        Rec r;
        ld_rec(rows + i, r);
        const double sc = score_state(h, 2, r.lo, r.hi & HI_KEY_MASK, r.aux, L, draws[i]);
        const uint64_t k = flip_f64((uint64_t)__double_as_longlong(sc));
        sk[i] = k;
        kmin = kmax = k;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
    }
    if ((threadIdx.x & 31) == 0 && kmin <= kmax) {
        atomicMin(&ctr->sk_min, (unsigned long long)kmin);
        atomicMax(&ctr->sk_max, (unsigned long long)kmax);
    }
}

__global__ void __launch_bounds__(TILE) score_rows_kernel(const Rec *__restrict__ rows, int64_t n, int h, int noise_mode,
                                                          ScoreLuts L, double *__restrict__ out,
                                                          const uint8_t *__restrict__ draws) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        Rec r;
        ld_rec(rows + i, r);
        out[i] = score_state(h, noise_mode, r.lo, r.hi & HI_KEY_MASK, r.aux, L, draws ? draws[i] : 50);
    }
}

// for every a[i] (sorted or not): number of elements of the ascending-sorted composite list b that
// are < a[i] (inclusive = 0) or <= a[i] (inclusive = 1); composite = (y, klo, khi) when words == 3
__device__ __forceinline__ bool comp_less(int words, int inclusive, uint64_t by, uint64_t bl, uint64_t bh, uint64_t y,
                                          uint64_t kl, uint64_t kh) {  // b < a (or b <= a)
    if (by != y) return by < y;
    if (words == 3) {
        if (bh != kh) return bh < kh;
        if (bl != kl) return bl < kl;
    }
    return inclusive;
}
__device__ __forceinline__ int64_t comp_lower(int words, int inclusive, const uint64_t *__restrict__ by,
                                              const uint64_t *__restrict__ bkl, const uint64_t *__restrict__ bkh, int64_t lo,
                                              int64_t hi, uint64_t y, uint64_t kl, uint64_t kh) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (comp_less(words, inclusive, by[mid], words == 3 ? bkl[mid] : 0, words == 3 ? bkh[mid] : 0, y, kl, kh)) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}
// out[i] (+)= #{ j : b[j] < a[i] } (or <=) for ascending-sorted b.  When a is ascending too (sorted_a), the CTA
// first brackets its slice of a inside b with two searches, so the per-element searches stay inside a short,
// cache-resident window instead of walking the whole list.
__global__ void __launch_bounds__(TILE) count_less_kernel(int words, int inclusive, const uint64_t *__restrict__ ay,
                                                          const uint64_t *__restrict__ akl, const uint64_t *__restrict__ akh,
                                                          int64_t na, const uint64_t *__restrict__ by,
                                                          const uint64_t *__restrict__ bkl, const uint64_t *__restrict__ bkh,
                                                          int64_t nb, int64_t *__restrict__ out, int accumulate, int sorted_a) {
    __shared__ int64_t s_lo, s_hi;
    const int64_t i0 = (int64_t)blockIdx.x * TILE, i = i0 + threadIdx.x;
    if (sorted_a) {
        if (threadIdx.x < 2) {
            const int64_t k = threadIdx.x == 0 ? i0 : min(i0 + TILE, na) - 1;
            const int64_t r = comp_lower(words, threadIdx.x == 0 ? 0 : 1, by, bkl, bkh, 0, nb, ay[k], words == 3 ? akl[k] : 0,
                                         words == 3 ? akh[k] : 0);
            if (threadIdx.x == 0) s_lo = r; else s_hi = r;
        }
        __syncthreads();
    }
    if (i >= na) return;
    const int64_t lo = sorted_a ? s_lo : 0, hi = sorted_a ? s_hi : nb;
    const int64_t r = comp_lower(words, inclusive, by, bkl, bkh, lo, hi, ay[i], words == 3 ? akl[i] : 0, words == 3 ? akh[i] : 0);
    out[i] = (accumulate ? out[i] : 0) + r;
}

// ---- owner partition specialised for <= 32 ranks: two kernels, keys read twice, no (digit, index) pairs
constexpr int PART_ITEMS = 8;                    // rows per thread; a warp owns 256 consecutive rows
constexpr int PART_TILE = TILE * PART_ITEMS;     // 2048 rows per CTA
__global__ void __launch_bounds__(TILE) owner_hist_kernel(const Rec *__restrict__ rows, int64_t n, uint32_t n_ranks,
                                                          uint32_t *__restrict__ matrix, uint32_t ntiles) {
    __shared__ uint32_t sh[32];
    if (threadIdx.x < 32) sh[threadIdx.x] = 0;
    __syncthreads();
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t wbase = (int64_t)blockIdx.x * PART_TILE + (int64_t)w * (32 * PART_ITEMS);
    uint32_t mine = 0;  // lane g accumulates the warp's count for owner g
#pragma unroll
    for (int q = 0; q < PART_ITEMS; ++q) {
        const int64_t i = wbase + q * 32 + lane;
        uint32_t o = 0xffffffffu;
        if (i < n) {
            uint64_t lo, hi;
            ld_cg_u64x2(reinterpret_cast<const uint64_t *>(rows + i), lo, hi);
            o = owner_of_key(lo, hi & HI_KEY_MASK, n_ranks);
        }
        for (uint32_t g = 0; g < n_ranks; ++g) {
            const uint32_t c = __popc(__ballot_sync(0xffffffffu, o == g));
            if (lane == g) mine += c;
        }
    }
    if (lane < n_ranks && mine) atomicAdd(&sh[lane], mine);
    __syncthreads();
    if (threadIdx.x < n_ranks) matrix[(uint64_t)threadIdx.x * ntiles + blockIdx.x] = sh[threadIdx.x];  // owner-major
}
__global__ void __launch_bounds__(TILE) owner_scatter_kernel(const Rec *__restrict__ rows, int64_t n, uint32_t n_ranks,
                                                             const uint32_t *__restrict__ matrix_scanned, uint32_t ntiles,
                                                             spl_key *__restrict__ send_keys, uint32_t *__restrict__ perm) {
    __shared__ uint32_t wcnt[TILE / 32][32];
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t wbase = (int64_t)blockIdx.x * PART_TILE + (int64_t)w * (32 * PART_ITEMS);
    uint64_t klo[PART_ITEMS], khi[PART_ITEMS];
    uint32_t own[PART_ITEMS];
    uint32_t mine = 0;
#pragma unroll
    for (int q = 0; q < PART_ITEMS; ++q) {
        const int64_t i = wbase + q * 32 + lane;
        own[q] = 0xffffffffu;
        if (i < n) {
            ld_cg_u64x2(reinterpret_cast<const uint64_t *>(rows + i), klo[q], khi[q]);
            own[q] = owner_of_key(klo[q], khi[q] & HI_KEY_MASK, n_ranks);
        }
        for (uint32_t g = 0; g < n_ranks; ++g) {
            const uint32_t c = __popc(__ballot_sync(0xffffffffu, own[q] == g));
            if (lane == g) mine += c;
        }
    }
    wcnt[w][lane] = lane < n_ranks ? mine : 0;
    __syncthreads();
    if (threadIdx.x < n_ranks) {  // exclusive over warps + the tile's global base for this owner
        uint32_t run = matrix_scanned[(uint64_t)threadIdx.x * ntiles + blockIdx.x];
        for (int ww = 0; ww < TILE / 32; ++ww) {
            const uint32_t c = wcnt[ww][threadIdx.x];
            wcnt[ww][threadIdx.x] = run;
            run += c;
        }
    }
    __syncthreads();
    uint32_t base = lane < n_ranks ? wcnt[w][lane] : 0;  // lane g holds the warp's running position for owner g
#pragma unroll
    for (int q = 0; q < PART_ITEMS; ++q) {
        const int64_t i = wbase + q * 32 + lane;
        uint32_t pos = 0;
        for (uint32_t g = 0; g < n_ranks; ++g) {
            const uint32_t bal = __ballot_sync(0xffffffffu, own[q] == g);
            const uint32_t b = __shfl_sync(0xffffffffu, base, g);
            if (own[q] == g) pos = b + __popc(bal & ((1u << lane) - 1));
            if (lane == g) base += __popc(bal);
        }
        if (i < n) {
            send_keys[pos].lo = klo[q];
            send_keys[pos].hi = khi[q];
            perm[pos] = (uint32_t)i;
        }
    }
}

// move every occupied slot of an old table into a larger one (tags preserved)
__global__ void __launch_bounds__(TILE) rehash_kernel(const uint64_t *__restrict__ old_table, uint64_t old_nb,
                                                      uint64_t *__restrict__ table, uint64_t nb, Counters *ctr) {
    const uint64_t s = (uint64_t)blockIdx.x * TILE + threadIdx.x;  // one thread per old slot
    if (s >= old_nb * BUCKET_SLOTS) return;
    uint64_t a, h;
    ld_cg_u64x2(bucket_key(old_table + ((s / BUCKET_SLOTS) << 3), (int)(s % BUCKET_SLOTS)), a, h);
    if ((a | h) == 0) return;
    uint64_t b = slot_of(hash_key(a, h & HI_KEY_MASK), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        for (int j = 0; j < BUCKET_SLOTS; ++j) {
            uint64_t oa, oh;
            cas128(bucket_key(table + (b << 3), j), 0, 0, a, h, oa, oh);
            if ((oa | oh) == 0) return;
        }
        if (++b == nb) b = 0;
    }
    atomicExch(&ctr->error, 1u);
}

}  // namespace spl
