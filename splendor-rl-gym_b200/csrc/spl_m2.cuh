// spl_m2.cuh -- card-set-grouped frontier expansion (the beam-search level of the speedrun solver).
//
// The visited set of State.solve (`trail`, src/solver.py:426, :447-450) is keyed by (cards, gems).  A level
// of the search touches few distinct card sets (about one per ten queue states, measured) and many gem
// hands per card set: a gem take keeps the card set, so the ~16 take successors of a parent and of every
// other parent with the same cards fall into ONE 2898-entry space (five gem counts 0..7, at most 10 in
// hand, src/gems.py:9,40-51).  This path therefore deduplicates per card set instead of per key:
//
//   visited set  = open-addressed table of 384-byte NODES, one per card set that was ever generated:
//                  {90-bit card mask, 2898-bit bitmap over the gem hands}  (`trail` membership = one bit)
//   one level    = 1. m2_count / m2_buys : per-parent fan-out; every card buy (it changes the card set) becomes
//                     one 8-byte sort item {target card-set hash, parent, card}; gem takes are NOT materialised
//                  2. LSD radix sort of {parents, buys} by the hash of their (target) card set
//                  3. m2_runs : boundaries of equal-hash runs + candidate-weight prefix
//                  4. m2_group_small / m2_group_big : one warp / one CTA per run loads the node, replays
//                     the takes of the run's parents and the run's buys (rebuilt from their parents' records)
//                     against an ON-CHIP table
//                     (min arrival index per gem hand, src/solver.py:447-450 first arrival wins), emits the
//                     winners with their scores and sets their bits.  No global atomics per candidate,
//                     no second visit to the table.
// Sorting by the hash that also selects the node makes the node accesses of a level monotone in memory.
// Winners are emitted in no particular order; link = parent_rank << 8 | ordinal carries the arrival
// order, and the beam cut breaks score ties on it (SPL_TIE_STABLE) or on the key (SPL_TIE_KEY).
#pragma once
#include "spl_kernels.cuh"

namespace spl {

constexpr int GEM_STATES = 2898;       // gem hands with every colour <= 7 and at most 10 gems
constexpr int NODE_BM_WORDS = 46;      // 2944 bits >= GEM_STATES
constexpr int NODE_WORDS = 48;         // 384 B = 6 DRAM bursts: {m0, m1 | OCC, bitmap[46]}
constexpr uint64_t NODE_OCC = 1ull << 63;
constexpr int SMALL_ITEMS = 32;        // runs handled by one warp: at most 32 items and SMALL_W candidates
constexpr int SMALL_W = 128;
constexpr int SM_TBL = 256;            // per-warp dedup slots (> SMALL_W, power of two)
constexpr int SM_STAGE = 48;           // per-warp winner staging (flushed above 16 entries)
struct GroupArgs;
constexpr int NUM_CLS = 8;             // run classes; used: CLS_WARP (one warp per run), CLS_CTA (one CTA per run)
constexpr int CLS_WARP = 6, CLS_CTA = 7;
constexpr int M2_WARPS = TILE / 32;
constexpr int BIG_DONE = 16;           // card sets of a run the CTA kernel remembers as done: it walks at most BIG_DONE + 1 per run
constexpr int BIG_AT_BITS = 24;        // item offset inside a run, packed under the arrival index in the CTA kernel's table
// Item id (low 32 bits of a sort item) of a round on one GPU: parent p of the round is id p, the buy of card `pos` (key
// bit) by parent p is ITEM_BUY | p << 7 | pos.  The buy is not stored anywhere else: the dedup kernels rebuild it from
// the parent's record (load_buy).  Every parent id (< np) is below every buy id.  Rounds of the card-set-sharded driver
// number their received buy records np + i instead.
constexpr int ITEM_PARENT_BITS = 24;   // parents of one round: at most 2^24 (splendor_b200.cu clamps chunk_parents to it)
constexpr uint32_t ITEM_BUY = 1u << 31;
__device__ __forceinline__ uint32_t buy_item_id(uint32_t p, int pos) { return ITEM_BUY | p << 7 | (uint32_t)pos; }

// card mask of a key as two words (90 bits)
__device__ __host__ __forceinline__ void mask_words(uint64_t lo, uint64_t hi, uint64_t &m0, uint64_t &m1) {
    m0 = (lo >> 15) | (hi << 49);
    m1 = (hi & HI_KEY_MASK) >> 15;
}
__device__ __host__ __forceinline__ uint64_t mask_hash(uint64_t m0, uint64_t m1) { return hash_key(m0, m1); }

// ------------------------------------------------------------------ node table
// find the node of card set (m0, m1) or claim an empty one (128-bit CAS on the header).  A card set is
// looked up by exactly one warp / CTA per round (all its candidates sit in one run), so nothing races
// on a node's bitmap; claims of the same empty slot by different card sets are settled by the CAS.
__device__ __forceinline__ uint64_t node_find_or_create(uint64_t *__restrict__ nodes, uint64_t nn, uint64_t m0, uint64_t m1,
                                                        bool &fresh, unsigned int *error) {
    const uint64_t want1 = m1 | NODE_OCC;
    uint64_t i = __umul64hi(mask_hash(m0, m1), nn);
    fresh = false;
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        uint64_t *N = nodes + i * NODE_WORDS;
        uint64_t a, b;
        ld_cg_u64x2(N, a, b);
        if (b == 0) {  // empty (an occupied header always carries NODE_OCC)
            cas128(N, 0, 0, m0, want1, a, b);
            if ((a | b) == 0) { fresh = true; return i; }
        }
        if (a == m0 && b == want1) return i;
        if (++i == nn) i = 0;
    }
    atomicExch(error, 2u);
    return 0;
}
__device__ __forceinline__ bool node_bit(const uint64_t *N, uint32_t r) {
    uint64_t w;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(w) : "l"(N + 2 + (r >> 6)));
    return (w >> (r & 63)) & 1;
}

// trail = {row: None for row in rows} (src/solver.py:426): one thread per row of the level-0 queue.  The host has
// checked that every row has a legal gem hand and that no two rows share a key.
__global__ void m2_root_kernel(uint64_t *nodes, uint64_t nn, const Rec *__restrict__ rows, int64_t n,
                               const uint16_t *__restrict__ gemrank, Counters *ctr) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint64_t lo = rows[t].lo, hi = rows[t].hi;
    uint64_t m0, m1;
    mask_words(lo, hi, m0, m1);
    bool fresh;
    const uint64_t i = node_find_or_create(nodes, nn, m0, m1, fresh, &ctr->error);
    const uint32_t r = gemrank[lo & GEM_MASK];
    atomicOr(reinterpret_cast<unsigned long long *>(nodes + i * NODE_WORDS + 2 + (r >> 6)), 1ull << (r & 63));
    if (fresh) atomicAdd(&ctr->n_new_nodes, 1u);
}

// move every node of an old table into a larger one: one warp per old slot
__global__ void __launch_bounds__(TILE) m2_rehash_kernel(const uint64_t *__restrict__ old_nodes, uint64_t old_nn,
                                                         uint64_t *__restrict__ nodes, uint64_t nn, Counters *ctr) {
    const uint64_t s = ((uint64_t)blockIdx.x * TILE + threadIdx.x) >> 5;
    const unsigned lane = threadIdx.x & 31;
    if (s >= old_nn) return;
    const uint64_t *O = old_nodes + s * NODE_WORDS;
    const uint64_t m1 = O[1];
    if (m1 == 0) return;
    uint64_t i = 0;
    if (lane == 0) {
        bool fresh;
        i = node_find_or_create(nodes, nn, O[0], m1 & ~NODE_OCC, fresh, &ctr->error);
    }
    i = __shfl_sync(0xffffffffu, i, 0);
    for (int w = lane; w < NODE_BM_WORDS; w += 32) nodes[i * NODE_WORDS + 2 + w] = O[2 + w];
}

// ------------------------------------------------------------------ 1. fan-out of the round's parents
// per parent: buys offset (exclusive scan), number of takes, sort key = high half of the card-set hash
__global__ void __launch_bounds__(TILE) m2_count_kernel(const Rec *__restrict__ front, int64_t np,
                                                        const DevTables *__restrict__ tabs,
                                                        const uint32_t *__restrict__ takes_idx,
                                                        uint32_t *__restrict__ boff, uint64_t *__restrict__ iv,
                                                        uint8_t *__restrict__ ntk8,
                                                        uint64_t *status, Counters *ctr, int ticket_id) {
    __shared__ SmemTabs s;
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    load_tabs(s, tabs);
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t p = (int64_t)tile * TILE + threadIdx.x;
    uint32_t nb = 0, ntk = 0;
    if (p < np) {
        Rec r;
        ld_rec(front + p, r);
        uint64_t bl, bh, m0, m1;
        uint32_t tk;
        derive_parent(s, takes_idx, r.lo, r.hi, r.aux, bl, bh, nb, tk);
        ntk = tk & 0xff;
        mask_words(r.lo, r.hi, m0, m1);
        iv[p] = (mask_hash(m0, m1) & 0xFFFFFFFF00000000ull) | (uint64_t)p;  // item = high half of the card-set hash << 32 | item id (ordered by its top 30 bits)
        ntk8[p] = (uint8_t)ntk;
    }
    uint32_t total, total_tk;
    block_excl_scan(ntk, warp_sums, total_tk);
    const uint32_t excl = block_excl_scan(nb, warp_sums, total);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, total, 0);
        if (threadIdx.x == 0) {
            s_base = e;
            if (total_tk) atomicAdd(&ctr->total_cands, (unsigned long long)total_tk);  // takes of the round
            if ((int64_t)(tile + 1) * TILE >= np) ctr->n_buys = e + total;
        }
    }
    __syncthreads();
    if (p < np) boff[p] = (uint32_t)(s_base + excl);
}

// card buys of the round's parents (src/solver.py:369-374) as items: high half of the hash of the child's card set
// (the parent's plus card `pos`) << 32 | buy_item_id(parent, pos), at np + boff[parent] + ordinal
struct BuySmem {
    SmemTabs tabs;
    uint64_t lo[TILE], hi[TILE];
    uint32_t prefb[TILE + 1];
    uint16_t blist[BUY_WIN];
    uint32_t warp_sums[TILE / 32 + 1];
};
__global__ void __launch_bounds__(TILE) m2_buys_kernel(const Rec *__restrict__ front, int64_t np,
                                                       const DevTables *__restrict__ tabs,
                                                       const uint32_t *__restrict__ takes_idx,
                                                       const uint32_t *__restrict__ boff, uint64_t *__restrict__ iv) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BuySmem &S = *reinterpret_cast<BuySmem *>(smem_raw);
    const unsigned tid = threadIdx.x;
    load_tabs(S.tabs, tabs);
    __syncthreads();
    const int64_t p0 = (int64_t)blockIdx.x * TILE, p = p0 + tid;
    const uint32_t b0 = boff[p0];
    uint64_t bm_lo = 0, bm_hi = 0;
    uint32_t nb = 0, tk = 0;
    if (p < np) {
        Rec r;
        ld_rec(front + p, r);
        derive_parent(S.tabs, takes_idx, r.lo, r.hi, r.aux, bm_lo, bm_hi, nb, tk);
        S.lo[tid] = r.lo; S.hi[tid] = r.hi;
    }
    uint32_t total_buys;
    const uint32_t prefb = block_excl_scan(nb, S.warp_sums, total_buys);
    S.prefb[tid] = prefb;
    if (tid == 0) S.prefb[TILE] = total_buys;
    for (uint32_t w0 = 0; w0 < total_buys; w0 += BUY_WIN) {
        __syncthreads();
        {
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
            uint64_t klo = S.lo[j], khi = S.hi[j], m0, m1;
            set_key_bit(klo, khi, pos);
            mask_words(klo, khi, m0, m1);
            const uint64_t g = (uint64_t)b0 + w0 + i;  // == boff[parent] + ordinal
            iv[np + g] = (mask_hash(m0, m1) & 0xFFFFFFFF00000000ull) | buy_item_id((uint32_t)(p0 + j), pos);
        }
    }
}

// ------------------------------------------------------------------ 2. sort of the packed items
// One stable LSD pass over 64-bit values (digit = bits shift..shift+7), tile = 4096 values per CTA.  Per-tile digit
// counts come from sort_hist_kernel + scan_u32_kernel (digit-major matrix).  The tile is first ordered by digit
// in shared memory, so that consecutive threads write consecutive addresses of each digit's output range (whole
// sectors) instead of scattering single values.
__global__ void __launch_bounds__(TILE, 4) psort_scatter_kernel(const uint64_t *__restrict__ v_in, int64_t n, int shift,
                                                                const uint32_t *__restrict__ matrix_scanned, uint32_t ntiles,
                                                                uint64_t *__restrict__ v_out) {
    __shared__ uint32_t whist[TILE / 32][SORT_BINS];
    __shared__ uint32_t dbase[SORT_BINS], gbase[SORT_BINS];
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint64_t stage[SORT_TILE];
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < (TILE / 32) * SORT_BINS; i += TILE) (&whist[0][0])[i] = 0;
    __syncthreads();
    const int64_t tbase = (int64_t)blockIdx.x * SORT_TILE, wbase = tbase + (int64_t)w * (32 * SORT_ITEMS);
    uint64_t v[SORT_ITEMS];
    uint16_t off[SORT_ITEMS];  // position of the value among the warp's values with the same digit (stable)
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {  // the warp's contiguous 512-value segment, 32 consecutive values per step
        const int64_t i = wbase + q * 32 + lane;
        const bool ok = i < n;
        v[q] = ok ? v_in[i] : 0;
        const uint32_t d = (uint32_t)(v[q] >> shift) & (SORT_BINS - 1);
        const unsigned act = __ballot_sync(0xffffffffu, ok);
        off[q] = 0;
        if (ok) {
            const unsigned peers = __match_any_sync(act, d);
            const int leader = __ffs(peers) - 1;
            uint32_t old = 0;
            if ((int)lane == leader) {
                old = whist[w][d];
                whist[w][d] = old + __popc(peers);
            }
            old = __shfl_sync(peers, old, leader);
            off[q] = (uint16_t)(old + __popc(peers & ((1u << lane) - 1)));
        }
        __syncwarp();
    }
    __syncthreads();
    {   // digit d = threadIdx.x: exclusive over warps; tile-local start of the digit; its global base for this tile
        const uint32_t d = threadIdx.x;
        uint32_t run = 0;
        for (int ww = 0; ww < TILE / 32; ++ww) {
            const uint32_t c = whist[ww][d];
            whist[ww][d] = run;
            run += c;
        }
        uint32_t tot;
        const uint32_t ex = block_excl_scan(run, warp_sums, tot);
        dbase[d] = ex;
        gbase[d] = matrix_scanned[(uint64_t)d * ntiles + blockIdx.x];
        for (int ww = 0; ww < TILE / 32; ++ww) whist[ww][d] += ex;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {  // stable placement inside the tile
        const int64_t i = wbase + q * 32 + lane;
        if (i < n) stage[whist[w][(uint32_t)(v[q] >> shift) & (SORT_BINS - 1)] + off[q]] = v[q];
    }
    __syncthreads();
    const uint32_t cnt = (uint32_t)min((int64_t)SORT_TILE, n - tbase);
    for (uint32_t i = threadIdx.x; i < cnt; i += TILE) {
        const uint64_t x = stage[i];
        const uint32_t d = (uint32_t)(x >> shift) & (SORT_BINS - 1);
        v_out[gbase[d] + (i - dbase[d])] = x;
    }
}

// ------------------------------------------------------------------ 2b. one-sweep passes (below 2^30 values)
// Stable LSD radix sort of 64-bit values (optionally with a 32-bit payload) by 10-bit digits.  One kernel reads the
// values once and builds the global histogram of every digit; each pass is then a single kernel: the tile (handed out
// by an atomic ticket) ranks its values, publishes its per-digit counts and finds its digit bases by a decoupled
// look-back over the tiles before it -- no per-pass histogram read, no scan launch.  status word (u32, one per tile
// and digit) = flag << 30 | count; flag 1 = tile count, 2 = inclusive prefix.
// The items of a round are ordered (and their runs are cut) by the top 30 bits of the card-set hash: three passes.
constexpr int ITEM_KEY_LO = 34;
constexpr int OS_BITS = 10, OS_BINS = 1 << OS_BITS, OS_MAX_PASSES = 7;
constexpr int OS_DPT = OS_BINS / TILE;          // digits per thread (4, consecutive)
static_assert(OS_DPT == 4, "the one-sweep pass moves the four digits of a thread as one 16-byte word");
constexpr int64_t OS_MAX_ITEMS = 1ll << 30;

// hist[p][d] += values whose digit p (bits lo_bit + 10 p ...) is d; dynamic shared memory: passes * OS_BINS words
__global__ void __launch_bounds__(TILE) os_hist_kernel(const uint64_t *__restrict__ v, int64_t n, int lo_bit, int passes,
                                                       uint32_t *__restrict__ hist) {
    extern __shared__ uint32_t os_sh[];
    for (int i = threadIdx.x; i < passes * OS_BINS; i += TILE) os_sh[i] = 0;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x; i < n; i += (int64_t)gridDim.x * TILE) {
        const uint64_t x = v[i] >> lo_bit;
        for (int p = 0; p < passes; ++p) atomicAdd(&os_sh[p * OS_BINS + ((uint32_t)(x >> (p * OS_BITS)) & (OS_BINS - 1))], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < passes * OS_BINS; i += TILE) {
        const uint32_t c = os_sh[i];
        if (c) atomicAdd(hist + i, c);
    }
}
// hist[p][d] -> exclusive prefix over d (one CTA of OS_BINS threads per pass)
__global__ void __launch_bounds__(OS_BINS) os_base_kernel(uint32_t *hist) {
    __shared__ uint32_t ws[OS_BINS / 32];
    uint32_t *h = hist + blockIdx.x * OS_BINS;
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t c = h[threadIdx.x];
    const uint32_t inc = warp_incl_scan(c);
    if (lane == 31) ws[w] = inc;
    __syncthreads();
    if (w == 0) {
        const uint32_t x = ws[lane], xi = warp_incl_scan(x);
        ws[lane] = xi - x;
    }
    __syncthreads();
    h[threadIdx.x] = inc - c + ws[w];
}

struct OsSmem {
    uint64_t stage[SORT_TILE];
    uint32_t gbase[OS_BINS];
    uint16_t whist[TILE / 32][OS_BINS];
    uint16_t dbase[OS_BINS];
    uint32_t warp_sums[TILE / 32 + 1];
    uint32_t tile;
    uint32_t stage_p[SORT_TILE];  // PAIR only (last member: the value-only launch leaves it out)
};
template <bool PAIR>
__global__ void __launch_bounds__(TILE, PAIR ? 3 : 4) os_scatter_kernel(const uint64_t *__restrict__ v_in, const uint32_t *__restrict__ p_in,
                                                                        int64_t n, int shift, const uint32_t *__restrict__ base /*[OS_BINS]*/,
                                                                        uint32_t *status, Counters *ctr, int ticket_id,
                                                                        uint64_t *__restrict__ v_out, uint32_t *__restrict__ p_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    OsSmem &S = *reinterpret_cast<OsSmem *>(smem_raw);
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) S.tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    for (int i = threadIdx.x; i < (TILE / 32) * OS_BINS / 2; i += TILE) reinterpret_cast<uint32_t *>(&S.whist[0][0])[i] = 0;
    __syncthreads();
    const uint32_t tile = S.tile;
    const int64_t tbase = (int64_t)tile * SORT_TILE, wbase = tbase + (int64_t)w * (32 * SORT_ITEMS);
    uint64_t v[SORT_ITEMS];
    uint32_t pl[PAIR ? SORT_ITEMS : 1];
    uint16_t off[SORT_ITEMS];  // position of the value among the warp's values with the same digit (stable)
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {
        const int64_t i = wbase + q * 32 + lane;
        v[q] = i < n ? v_in[i] : 0;
        if (PAIR) pl[q] = i < n ? p_in[i] : 0;
    }
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {
        const bool ok = wbase + q * 32 + lane < n;
        const uint32_t d = (uint32_t)(v[q] >> shift) & (OS_BINS - 1);
        const unsigned act = __ballot_sync(0xffffffffu, ok);
        off[q] = 0;
        if (ok) {
            const unsigned peers = __match_any_sync(act, d);
            const int leader = __ffs(peers) - 1;
            uint32_t old = 0;
            if ((int)lane == leader) {
                old = S.whist[w][d];
                S.whist[w][d] = (uint16_t)(old + __popc(peers));
            }
            old = __shfl_sync(peers, old, leader);
            off[q] = (uint16_t)(old + __popc(peers & ((1u << lane) - 1)));
        }
        __syncwarp();
    }
    __syncthreads();
    // digits 4t..4t+3 of thread t: exclusive over warps, tile count -> published; tile-local start of each digit
    const uint32_t d0 = threadIdx.x * OS_DPT;
    uint32_t cnt[OS_DPT] = {0, 0, 0, 0};
    for (int ww = 0; ww < TILE / 32; ++ww) {
        uint2 x = *reinterpret_cast<uint2 *>(&S.whist[ww][d0]);
        const uint32_t c0 = x.x & 0xffffu, c1 = x.x >> 16, c2 = x.y & 0xffffu, c3 = x.y >> 16;
        x.x = cnt[0] | (cnt[1] << 16); x.y = cnt[2] | (cnt[3] << 16);
        *reinterpret_cast<uint2 *>(&S.whist[ww][d0]) = x;
        cnt[0] += c0; cnt[1] += c1; cnt[2] += c2; cnt[3] += c3;
    }
    constexpr uint32_t VAL = (1u << 30) - 1;
    uint32_t *mine = status + (uint64_t)tile * OS_BINS + d0;
    {
        const uint32_t f = tile == 0 ? 2u << 30 : 1u << 30;
        uint4 a{f | cnt[0], f | cnt[1], f | cnt[2], f | cnt[3]};
        asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(mine), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w) : "memory");
    }
    {
        uint32_t tot;
        const uint32_t ex = block_excl_scan(cnt[0] + cnt[1] + cnt[2] + cnt[3], S.warp_sums, tot);
        const uint32_t e0 = ex, e1 = e0 + cnt[0], e2 = e1 + cnt[1], e3 = e2 + cnt[2];
        *reinterpret_cast<uint2 *>(&S.dbase[d0]) = uint2{e0 | (e1 << 16), e2 | (e3 << 16)};
        for (int ww = 0; ww < TILE / 32; ++ww) {  // tile-local position = digit start + warps before + rank in warp
            uint2 x = *reinterpret_cast<uint2 *>(&S.whist[ww][d0]);
            x.x += e0 | (e1 << 16); x.y += e2 | (e3 << 16);  // all sums <= 4096: the halves never carry
            *reinterpret_cast<uint2 *>(&S.whist[ww][d0]) = x;
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < SORT_ITEMS; ++q) {  // stable placement inside the tile
        if (wbase + q * 32 + lane < n) {
            const uint32_t at = S.whist[w][(uint32_t)(v[q] >> shift) & (OS_BINS - 1)] + off[q];
            S.stage[at] = v[q];
            if (PAIR) S.stage_p[at] = pl[q];
        }
    }
    // look-back over the tiles before this one (they hold earlier tickets, so they are resident or finished)
    uint32_t ex[OS_DPT] = {0, 0, 0, 0};
    if (tile > 0) {
        unsigned open = 15;  // digits whose walk has not met an inclusive prefix yet
        for (int64_t p = (int64_t)tile - 1; open; --p) {
            const uint32_t *src = status + (uint64_t)p * OS_BINS + d0;
            uint32_t s[OS_DPT];
            bool ready;
            do {
                asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(s[0]), "=r"(s[1]), "=r"(s[2]), "=r"(s[3]) : "l"(src) : "memory");
                ready = true;
#pragma unroll
                for (int k = 0; k < OS_DPT; ++k) ready = ready && (!((open >> k) & 1) || (s[k] >> 30) != 0);
            } while (!ready);
#pragma unroll
            for (int k = 0; k < OS_DPT; ++k)
                if ((open >> k) & 1) {
                    ex[k] += s[k] & VAL;
                    if ((s[k] >> 30) == 2) open &= ~(1u << k);
                }
        }
        const uint32_t f = 2u << 30;
        asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(mine), "r"(f | (ex[0] + cnt[0])), "r"(f | (ex[1] + cnt[1])),
                     "r"(f | (ex[2] + cnt[2])), "r"(f | (ex[3] + cnt[3])) : "memory");
    }
    {
        const uint4 b = *reinterpret_cast<const uint4 *>(base + d0);
        *reinterpret_cast<uint4 *>(&S.gbase[d0]) = uint4{b.x + ex[0], b.y + ex[1], b.z + ex[2], b.w + ex[3]};
    }
    __syncthreads();
    const uint32_t cnt_tile = (uint32_t)min((int64_t)SORT_TILE, n - tbase);
    for (uint32_t i = threadIdx.x; i < cnt_tile; i += TILE) {
        const uint64_t x = S.stage[i];
        const uint32_t d = (uint32_t)(x >> shift) & (OS_BINS - 1);
        const uint32_t to = S.gbase[d] + (i - S.dbase[d]);
        v_out[to] = x;
        if (PAIR) p_out[to] = S.stage_p[i];
    }
}

// ------------------------------------------------------------------ 3. runs of equal sort key
// run_start[r] = first sorted item of run r, run_wpre[r] = candidates (takes of parents + buy records)
// in the runs before r.  Two look-back chains (run count, weight) walked by two warps at once.
constexpr int RUN_ITEMS = 8;
__global__ void __launch_bounds__(TILE) m2_runs_kernel(const uint64_t *__restrict__ iv, int64_t n_items, uint32_t np,
                                                       const uint8_t *__restrict__ ntk8,
                                                       uint32_t *__restrict__ run_start, uint32_t *__restrict__ run_wpre,
                                                       uint64_t *status_f, uint64_t *status_w, Counters *ctr, int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_fbase, s_wbase;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * RUN_ITEMS;
    uint32_t flags = 0, w[RUN_ITEMS], fsum = 0, wsum = 0;
    uint64_t prev = (b0 > 0 && b0 - 1 < n_items) ? iv[b0 - 1] >> ITEM_KEY_LO : 0;
#pragma unroll
    for (int q = 0; q < RUN_ITEMS; ++q) {
        const int64_t i = b0 + q;
        w[q] = 0;
        if (i < n_items) {
            const uint64_t v = iv[i], k = v >> ITEM_KEY_LO;
            if (i == 0 || k != prev) { flags |= 1u << q; ++fsum; }
            prev = k;
            const uint32_t id = (uint32_t)v;
            w[q] = id < np ? ntk8[id] : 1u;
            wsum += w[q];
        }
    }
    // tile totals: runs <= 2048 (12 bits), weight <= 2048 * 100 (18 bits): one packed scan
    uint32_t tot;
    const uint32_t ex = block_excl_scan(wsum << 12 | fsum, warp_sums, tot);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status_f, tile, tot & 0xfffu, 0);
        if (threadIdx.x == 0) s_fbase = e;
    } else if (threadIdx.x < 64) {
        const uint64_t e = lookback_exclusive(status_w, tile, tot >> 12, 0);
        if (threadIdx.x == 32) s_wbase = e;
    }
    __syncthreads();
    uint64_t r = s_fbase + (ex & 0xfffu), wp = s_wbase + (ex >> 12);
#pragma unroll
    for (int q = 0; q < RUN_ITEMS; ++q) {
        if (flags >> q & 1) {
            run_start[r] = (uint32_t)(b0 + q);
            run_wpre[r] = (uint32_t)wp;
            ++r;
        }
        wp += w[q];
    }
    if (b0 <= n_items - 1 && n_items - 1 < b0 + RUN_ITEMS) {  // the thread that owns the last item: sentinel
        run_start[r] = (uint32_t)n_items;
        run_wpre[r] = (uint32_t)wp;
        ctr->n_runs = (unsigned int)r;
    }
}

// ------------------------------------------------------------------ 4. per-run dedup
struct GroupArgs {
    const Rec *front;              // the round's parents (rank order)
    const Rec *brec;               // the buy records the round received (card-set-sharded driver; one GPU: none)
    const uint64_t *iv;            // sorted items: hash half << 32 | item id (id < np: parent; else a buy, see ITEM_BUY)
    const uint32_t *run_start, *run_wpre;
    uint32_t np;
    int64_t rank_base;             // global rank of parent 0 of the round (when the parents' ranks are contiguous) ...
    const uint64_t *grank;         // ... or the global rank of every parent of the round (sharded queue), ascending
    int unordered;                 // buy records are not in arrival order (received from several ranks)
    uint32_t warp_max;             // runs of more candidates than this go to the CTA kernel
    const DevTables *tabs;
    const uint32_t *takes_idx;
    const uint16_t *takes_edges;
    const uint16_t *gemrank;
    const uint16_t *rankgems;      // inverse of gemrank: [GEM_STATES] gem hand of a dense index
    uint64_t *nodes;
    uint64_t nn;
    // Output: winners (any order; link carries the arrival order) and their order-preserving score keys, appended
    // densely at out_base + ctr->n_emitted (reserved in batches: per CTA / per 17..48 staged records / per run)
    Rec *out;
    uint64_t *out_sk;
    uint64_t out_base;
    uint32_t *cls_list[NUM_CLS];   // run lists per candidate-count class (m2_dispatch_kernel)
    int h, noise_mode;
    ScoreLuts L;
    Counters *ctr;
};

// ---- warp kernel: one warp per run.  The candidates of a run are visited in ARRIVAL ORDER, so "first arrival
// wins" (src/solver.py:447-450) needs nothing but the node's bitmap: a candidate whose bit is clear is the first
// arrival of its gem hand (it sets the bit), every later one finds the bit set.  Arrival order inside a run:
//   * the run's parents are in rank order and its buy records in (generating parent, ordinal) order -- the sort is
//     stable and both were generated in that order;
//   * all takes of a parent P carry t = P << 8 | ordinal, a buy record carries t = Q << 8 | ordinal of its
//     generating parent Q, and Q != P for every parent P of the run (Q owns one card less than the run's card
//     set), so merging the two lists by rank alone yields the arrival order.
__device__ __forceinline__ uint32_t item_id(const GroupArgs &A, uint32_t i) { return (uint32_t)A.iv[i]; }
__device__ __forceinline__ uint64_t parent_rank(const GroupArgs &A, uint32_t id) {
    return A.grank ? A.grank[id] : (uint64_t)(A.rank_base + id);
}
// the buy record {child key, child aux, link = parent rank << 8 | ordinal} of item id `id` (>= np): as received
// (UNORDERED), or rebuilt from the record of the parent and the card named in the id
template <bool UNORDERED>
__device__ __forceinline__ void load_buy(const GroupArgs &A, const SmemTabs &tabs, uint32_t id, Rec &b) {
    if (UNORDERED) {
        ld_rec(A.brec + (id - A.np), b);
        return;
    }
    const uint32_t p = (id >> 7) & ((1u << ITEM_PARENT_BITS) - 1);
    const int pos = id & 127;
    Rec par;
    ld_rec(A.front + p, par);
    buy_child(tabs, par.lo, par.hi, par.aux, pos, b.lo, b.hi, b.aux);
    uint64_t bl, bh;
    buy_mask(tabs, par.lo, par.hi, par.aux, bl, bh);
    b.link = (uint64_t)(A.rank_base + p) << 8 | buy_ordinal(bl, bh, pos);
}
// only the key words {lo, hi} of buy item `id` (the thread kernel's first look at a run)
template <bool UNORDERED>
__device__ __forceinline__ void load_buy_key(const GroupArgs &A, const SmemTabs &tabs, uint32_t id, uint64_t &lo, uint64_t &hi) {
    if (UNORDERED) {
        ld_cg_u64x2(reinterpret_cast<const uint64_t *>(A.brec + (id - A.np)), lo, hi);
        return;
    }
    Rec b;
    load_buy<false>(A, tabs, id, b);
    lo = b.lo;
    hi = b.hi;
}

// per-warp winner staging: records are collected in shared memory and written out 17..48 at a time behind one
// global atomic (dense output, few same-address atomics)
constexpr int M2_WARPS_ = TILE / 32;
struct WarpStage {
    uint64_t *st;                        // this warp's slice of st[5][warps][SM_STAGE] in shared memory: one pointer, the
    uint32_t cnt;                        // five columns sit at compile-time strides (cnt: warp-uniform)
    uint64_t kmin, kmax;
    __device__ __forceinline__ uint64_t &lo(uint32_t i) const { return st[i]; }
    __device__ __forceinline__ uint64_t &hi(uint32_t i) const { return st[1 * M2_WARPS_ * SM_STAGE + i]; }
    __device__ __forceinline__ uint64_t &aux(uint32_t i) const { return st[2 * M2_WARPS_ * SM_STAGE + i]; }
    __device__ __forceinline__ uint64_t &link(uint32_t i) const { return st[3 * M2_WARPS_ * SM_STAGE + i]; }
    __device__ __forceinline__ uint64_t &sk(uint32_t i) const { return st[4 * M2_WARPS_ * SM_STAGE + i]; }
};
__device__ __forceinline__ void stage_flush(const GroupArgs &A, WarpStage &W) {
    const unsigned lane = threadIdx.x & 31;
    __syncwarp();
    uint64_t base = 0;
    if (lane == 0) base = atomicAdd(&A.ctr->n_emitted, (unsigned long long)W.cnt);
    base = __shfl_sync(0xffffffffu, base, 0) + A.out_base;
    for (uint32_t i = lane; i < W.cnt; i += 32) {
        Rec r{W.lo(i), W.hi(i), W.aux(i), W.link(i)};
        st_rec(A.out + base + i, r);
        if (A.out_sk) A.out_sk[base + i] = W.sk(i);
    }
    W.cnt = 0;
    __syncwarp();
}

// Open the node of card set (M0, M1) for this warp: the whole 384-byte node at the home slot is fetched in one
// round trip (header + bitmap, 48 words over the lanes); if the home slot holds the set, or is empty and this warp
// claims it, nothing else is read.  bm[0..45] (shared memory of the warp) receives the bitmap.
__device__ __forceinline__ uint64_t *node_open(const GroupArgs &A, uint64_t M0, uint64_t M1, uint64_t *bm, uint32_t &n_fresh) {
    const unsigned lane = threadIdx.x & 31;
    uint64_t i = __umul64hi(mask_hash(M0, M1), A.nn);
    const uint64_t *H = A.nodes + i * NODE_WORDS;
    uint64_t w0, w1 = 0;
    asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(w0) : "l"(H + lane));
    if (lane < 16) asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(w1) : "l"(H + 32 + lane));
    uint64_t h0 = __shfl_sync(0xffffffffu, w0, 0), h1 = __shfl_sync(0xffffffffu, w0, 1);
    int state = 0;  // 0: another set lives here (probe on), 1: found, 2: claimed now (fresh)
    if (lane == 0) {
        if (h1 == 0) {
            cas128(A.nodes + i * NODE_WORDS, 0, 0, M0, M1 | NODE_OCC, h0, h1);
            if ((h0 | h1) == 0) state = 2;
        }
        if (state == 0 && h0 == M0 && h1 == (M1 | NODE_OCC)) state = 1;
    }
    state = __shfl_sync(0xffffffffu, state, 0);
    if (state == 0) {  // collision at the home slot: ordinary probe sequence, then fetch that node's bitmap
        int fresh_i = 0;
        if (lane == 0) {
            bool fresh;
            i = node_find_or_create(A.nodes, A.nn, M0, M1, fresh, &A.ctr->error);
            fresh_i = fresh;
        }
        i = __shfl_sync(0xffffffffu, i, 0);
        state = __shfl_sync(0xffffffffu, fresh_i, 0) ? 2 : 1;
        if (state == 1) {
            H = A.nodes + i * NODE_WORDS;
            asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(w0) : "l"(H + lane));
            if (lane < 16) asm volatile("ld.global.cg.u64 %0, [%1];" : "=l"(w1) : "l"(H + 32 + lane));
        }
    }
    if (state == 2) { w0 = 0; w1 = 0; if (lane == 0) ++n_fresh; }
    if (lane >= 2) bm[lane - 2] = w0;
    if (lane < 16) bm[30 + lane] = w1;
    __syncwarp();
    return A.nodes + i * NODE_WORDS;
}
__device__ __forceinline__ void node_close(uint64_t *N, const uint64_t *bm) {
    const unsigned lane = threadIdx.x & 31;
    __syncwarp();
    if (lane >= 2) N[lane] = bm[lane - 2];
    if (lane < 16) N[32 + lane] = bm[30 + lane];
}

// One step of the arrival-ordered walk: up to 32 candidates (act lanes), EARLIER arrivals on lower lanes.  `dups`:
// several lanes may carry the same gem hand (buy records of different parents), then the lowest lane speaks for it.
// A candidate wins iff its bit was clear; winners are staged with their scores.  Called by all 32 lanes.
__device__ __forceinline__ void bm_step(const GroupArgs &A, WarpStage &W, uint64_t *bm, bool act, bool dups, uint32_t g,
                                        uint64_t t, uint64_t clo, uint64_t chi, uint64_t caux) {
    const unsigned lane = threadIdx.x & 31;
    uint32_t rk = 0;
    if (act) rk = __ldg(A.gemrank + g);
    bool lead = act;
    if (dups) {
        const unsigned m = __ballot_sync(0xffffffffu, act);
        if (act) lead = lane == (unsigned)(__ffs(__match_any_sync(m, rk)) - 1);
    }
    bool win = false;
    if (lead) {
        // (64-bit OR on shared memory compiles to a CAS loop, a quarter of this kernel's instructions; the native 32-bit
        // ATOMS.OR with a returned value was measured and is slower here: 97 vs 78 ms per beam-30M solve)
        // Most candidates are duplicates: a set bit is final, so only clear ones pay for the atomic.
        const unsigned long long bit = 1ull << (rk & 63);
        if (!(bm[rk >> 6] & bit)) win = !(atomicOr(reinterpret_cast<unsigned long long *>(&bm[rk >> 6]), bit) & bit);
    }
    const unsigned wb = __ballot_sync(0xffffffffu, win);
    if (win) {
        const uint32_t at = W.cnt + __popc(wb & ((1u << lane) - 1));
        W.lo(at) = clo; W.hi(at) = chi; W.aux(at) = caux; W.link(at) = t;
        if (A.out_sk) {
            const uint64_t k = flip_f64((uint64_t)__double_as_longlong(score_state(A.h, A.noise_mode, clo, chi & HI_KEY_MASK, caux, A.L)));
            W.sk(at) = k;
            W.kmin = min(W.kmin, k); W.kmax = max(W.kmax, k);
        }
    }
    W.cnt += __popc(wb);
    if (W.cnt > SM_STAGE - 32) stage_flush(A, W);
}
// the gem takes of TWO parents in one step: lanes 0..15 the earlier parent (lane P0 of the item window), lanes 16..31
// the later one (lane P1); both have at most 16 takes.  Their successors may coincide, so the step resolves equal
// gem hands in lane order (== arrival order).
__device__ __forceinline__ void take_steps_pair(const GroupArgs &A, WarpStage &W, uint64_t *bm, const Rec &it, uint64_t grank,
                                                uint32_t tk, uint32_t nb, int P0, int P1) {
    const unsigned lane = threadIdx.x & 31;
    const int src = lane < 16 ? P0 : P1;
    const uint64_t plo = __shfl_sync(0xffffffffu, it.lo, src), phi = __shfl_sync(0xffffffffu, it.hi, src);
    const uint64_t paux = __shfl_sync(0xffffffffu, it.aux, src), pgr = __shfl_sync(0xffffffffu, grank, src);
    const uint32_t ptk = __shfl_sync(0xffffffffu, tk, src), pnb = __shfl_sync(0xffffffffu, nb, src);
    const uint32_t q = lane & 15;
    const bool act = q < (ptk & 0xff);
    const uint32_t g = act ? (uint32_t)__ldg(A.takes_edges + (ptk >> 8) + q) : 0u;
    bm_step(A, W, bm, act, true, g, (pgr << 8) | (pnb + q), (plo & ~GEM_MASK) | g, phi, paux);
}
// the gem takes (src/solver.py:381-388) of one parent (fields warp-uniform), 32 table edges per step
__device__ __forceinline__ void take_steps(const GroupArgs &A, WarpStage &W, uint64_t *bm, uint64_t plo, uint64_t phi, uint64_t paux,
                                           uint64_t pgr, uint32_t ptk, uint32_t pnb) {
    const unsigned lane = threadIdx.x & 31;
    const uint32_t ntk = ptk & 0xff;
    for (uint32_t q0 = 0; q0 < ntk; q0 += 32) {
        const uint32_t q = q0 + lane;
        const bool act = q < ntk;
        const uint32_t g = act ? (uint32_t)__ldg(A.takes_edges + (ptk >> 8) + q) : 0u;
        bm_step(A, W, bm, act, false, g, (pgr << 8) | (pnb + q), (plo & ~GEM_MASK) | g, phi, paux);
    }
}
// parent item `i` of the sorted list -> record, fan-out, rank, card-set words
__device__ __forceinline__ void load_parent_item(const GroupArgs &A, const SmemTabs &tabs, uint32_t i, Rec &it, uint32_t &nb,
                                                 uint32_t &tk, uint64_t &grank, uint64_t &m0, uint64_t &m1) {
    const uint32_t id = item_id(A, i);
    ld_rec(A.front + id, it);
    uint64_t bl, bh;
    derive_parent(tabs, A.takes_idx, it.lo, it.hi, it.aux, bl, bh, nb, tk);
    grank = parent_rank(A, id);
    mask_words(it.lo, it.hi, m0, m1);
}
__device__ __forceinline__ void warp_epilogue(const GroupArgs &A, WarpStage &W, uint32_t n_fresh) {
    const unsigned lane = threadIdx.x & 31;
    if (W.cnt) stage_flush(A, W);
    if (lane == 0 && n_fresh) atomicAdd(&A.ctr->n_new_nodes, n_fresh);
    if (A.out_sk) {
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            W.kmin = min(W.kmin, __shfl_xor_sync(0xffffffffu, W.kmin, d));
            W.kmax = max(W.kmax, __shfl_xor_sync(0xffffffffu, W.kmax, d));
        }
        if (lane == 0 && W.kmin <= W.kmax) {
            atomicMin(&A.ctr->sk_min, (unsigned long long)W.kmin);
            atomicMax(&A.ctr->sk_max, (unsigned long long)W.kmax);
        }
    }
}

#ifndef SPL_WARP_BATCH
#define SPL_WARP_BATCH 8  // measured per beam-30M solve: 1: 290, 2: 267, 4: 257, 8: 254, 16: 268, 32: 262, 64: 276 ms
#endif
constexpr int WARP_BATCH = SPL_WARP_BATCH; // runs a warp of the warp kernel draws per ticket
constexpr int MAX_SETS = 4;  // card sets of a run the warp kernel remembers as done: it walks at most MAX_SETS + 1 per run
constexpr int BSORT_MAX = 512;  // buy records of one run the warp kernel can put into arrival order itself
struct WarpSmem {
    SmemTabs tabs;
    uint64_t bm[M2_WARPS][NODE_BM_WORDS + 2];
    uint64_t st[5][M2_WARPS][SM_STAGE];  // lo, hi, aux, link, sk
    uint64_t done[M2_WARPS][MAX_SETS][2]; // card sets of the current run walked so far (rarely more than one)
    uint64_t bsort[M2_WARPS][BSORT_MAX]; // UNORDERED only (last member: the arrival-ordered launch leaves it out)
};

// Class CLS_WARP of the dispatch (THREAD_W < candidates <= WARP_W): one warp per run.  The run is streamed through a
// parent window and a buy-record window of 32 lanes each, once per card set it holds (almost always one; several
// only when two sets share a 30-bit sort key).  Persistent grid: warps draw batches of list entries from a ticket.
#ifndef SPL_WARP_CTAS
#define SPL_WARP_CTAS 4  // resident CTAs per SM of the warp kernel (64 registers per thread; 3 and 5 measured slower)
#endif
template <bool UNORDERED>
__global__ void __launch_bounds__(TILE, SPL_WARP_CTAS) m2_group_warp_kernel(GroupArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    WarpSmem &S = *reinterpret_cast<WarpSmem *>(smem_raw);
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    load_tabs(S.tabs, A.tabs);
    __syncthreads();
    uint64_t *bm = S.bm[w];
    WarpStage W{S.st[0][w], 0, ~0ull, 0};
    const uint32_t n_list = A.ctr->n_cls[CLS_WARP];
    uint32_t n_fresh = 0;
    // Runs weigh 17 .. 1024 candidates and their order in the list is whatever the dispatch kernel's atomics made it:
    // warps draw batches of WARP_BATCH runs from a ticket (the next batch's ticket is in flight while this one is
    // walked) instead of striding over the list, so the launch ends when the work does, not with its unluckiest warp.
    uint32_t next_base = 0;
    if (lane == 0) next_base = atomicAdd(&A.ctr->ticket[2], (unsigned)WARP_BATCH);
    for (;;) {
        const uint32_t base = __shfl_sync(0xffffffffu, next_base, 0);
        if (base >= n_list) break;
        if (lane == 0) next_base = atomicAdd(&A.ctr->ticket[2], (unsigned)WARP_BATCH);
        const uint32_t j_end = min(base + (uint32_t)WARP_BATCH, n_list);
      for (uint32_t j = base; j < j_end; ++j) {
        const uint32_t r = A.cls_list[CLS_WARP][j];
        const uint32_t s = A.run_start[r], e = A.run_start[r + 1];
        // parents [s, pe), buy records [pe, e)
        uint32_t pe = s;
        for (uint32_t b0 = s; b0 < e; b0 += 32) {
            const unsigned pm = __ballot_sync(0xffffffffu, b0 + lane < e && item_id(A, b0 + lane) < A.np);
            pe += __popc(pm);
            if (pm != 0xffffffffu) break;
        }
        // Records that came from several ranks are not in arrival order: sort this run's (link, index) pairs in shared
        // memory (bitonic, warp-cooperative) and read the buy window through the sorted indices.
        const uint32_t nbuy = e - pe;
        const bool resort = UNORDERED && nbuy > 1;
        uint64_t *bs = S.bsort[w];
        if (resort) {
            if (nbuy > BSORT_MAX) {  // (cannot happen while warp_max <= BSORT_MAX; kept as a guard)
                if (lane == 0) A.cls_list[CLS_CTA][atomicAdd(&A.ctr->n_cls[CLS_CTA], 1u)] = r;
                continue;
            }
            uint32_t npow = 32;
            while (npow < nbuy) npow <<= 1;
            for (uint32_t i = lane; i < npow; i += 32)
                bs[i] = i < nbuy ? (A.brec[item_id(A, pe + i) - A.np].link << 10) | i : ~0ull;
            __syncwarp();
            for (uint32_t k = 2; k <= npow; k <<= 1)
                for (uint32_t jj = k >> 1; jj > 0; jj >>= 1) {
                    for (uint32_t i = lane; i < npow; i += 32) {
                        const uint32_t x = i ^ jj;
                        if (x > i) {
                            const uint64_t a = bs[i], b = bs[x];
                            if ((a > b) == ((i & k) == 0)) { bs[i] = b; bs[x] = a; }
                        }
                    }
                    __syncwarp();
                }
        }
        uint64_t (*done)[2] = S.done[w];  // card sets done so far (shared memory: keeps 16 registers out of the walk)
        int n_done = 0;
        uint32_t lead = s;
        while (lead != 0xFFFFFFFFu) {
            uint64_t M0 = 0, M1 = 0;
            if (lane == 0) {
                const uint32_t id = item_id(A, lead);
                Rec src;
                if (id < A.np) ld_rec(A.front + id, src); else load_buy<UNORDERED>(A, S.tabs, id, src);
                mask_words(src.lo, src.hi, M0, M1);
            }
            M0 = __shfl_sync(0xffffffffu, M0, 0); M1 = __shfl_sync(0xffffffffu, M1, 0);
            uint64_t *N = node_open(A, M0, M1, bm, n_fresh);
            uint32_t next_lead = 0xFFFFFFFFu;
            Rec it{0, 0, 0, 0}, bt{0, 0, 0, 0};
            uint32_t nb = 0, tk = 0;
            uint64_t grank = 0, brank = 0;
            uint32_t bnext = pe, pnext = s;   // first item not loaded into a window yet
            unsigned bmask = 0, pmask = 0;
            for (;;) {
                if (!pmask && pnext < pe) {  // refill the parent window
                    const bool valid = pnext + lane < pe;
                    uint64_t m0 = 0, m1 = 0;
                    if (valid) load_parent_item(A, S.tabs, pnext + lane, it, nb, tk, grank, m0, m1);
                    const bool ok = valid && m0 == M0 && m1 == M1;
                    bool other = valid && !ok;  // a card set not walked yet?
#pragma unroll
                    for (int d = 0; d < MAX_SETS; ++d) other = other && !(d < n_done && done[d][0] == m0 && done[d][1] == m1);
                    const unsigned om = __ballot_sync(0xffffffffu, other);
                    if (om) next_lead = min(next_lead, pnext + (uint32_t)__ffs(om) - 1);
                    pmask = __ballot_sync(0xffffffffu, ok);
                    pnext += 32;
                    continue;
                }
                if (!bmask && bnext < e) {  // refill the buy window
                    const bool valid = bnext + lane < e;
                    uint64_t m0 = 0, m1 = 0;
                    if (valid) {
                        const uint32_t at = resort ? pe + (uint32_t)(bs[bnext - pe + lane] & 1023u) : bnext + lane;
                        load_buy<UNORDERED>(A, S.tabs, item_id(A, at), bt);
                        mask_words(bt.lo, bt.hi, m0, m1);
                        brank = bt.link >> 8;
                    }
                    const bool ok = valid && m0 == M0 && m1 == M1;
                    bool other = valid && !ok;
#pragma unroll
                    for (int d = 0; d < MAX_SETS; ++d) other = other && !(d < n_done && done[d][0] == m0 && done[d][1] == m1);
                    const unsigned om = __ballot_sync(0xffffffffu, other);
                    if (om) {  // item position of the first record of a card set not walked yet
                        const uint32_t j = bnext - pe + (uint32_t)__ffs(om) - 1;
                        next_lead = min(next_lead, resort ? pe + (uint32_t)(bs[j] & 1023u) : pe + j);
                    }
                    bmask = __ballot_sync(0xffffffffu, ok);
                    bnext += 32;
                    continue;
                }
                if (!pmask && !bmask) break;
                const uint64_t X = pmask ? __shfl_sync(0xffffffffu, grank, __ffs(pmask) - 1) : ~0ull;
                const unsigned m = bmask & __ballot_sync(0xffffffffu, brank < X);
                if (m) {  // the buy records of the window that arrive before the next parent
                    bm_step(A, W, bm, (m >> lane) & 1, true, (uint32_t)(bt.lo & GEM_MASK), bt.link, bt.lo, bt.hi, bt.aux);
                    bmask &= ~m;
                } else {  // pmask != 0 here: every record left in the window arrives after parent X
                    const int P = __ffs(pmask) - 1;
                    pmask &= pmask - 1;
                    // the next parent of the window rides along if both have at most 16 takes and no buy record arrives
                    // between them (none left in the window with a smaller rank, none outside the window at all)
                    const int P1 = pmask ? __ffs(pmask) - 1 : -1;
                    bool pair = false;
                    if (P1 >= 0) {
                        const uint32_t n0 = __shfl_sync(0xffffffffu, tk, P) & 0xff, n1 = __shfl_sync(0xffffffffu, tk, P1) & 0xff;
                        const uint64_t X1 = __shfl_sync(0xffffffffu, grank, P1);
                        const unsigned between = bmask & __ballot_sync(0xffffffffu, brank < X1);
                        pair = n0 <= 16 && n1 <= 16 && between == 0 && (bmask != 0 || bnext >= e);
                    }
                    if (pair) {
                        pmask &= pmask - 1;
                        take_steps_pair(A, W, bm, it, grank, tk, nb, P, P1);
                    } else {
                        take_steps(A, W, bm, __shfl_sync(0xffffffffu, it.lo, P), __shfl_sync(0xffffffffu, it.hi, P),
                                   __shfl_sync(0xffffffffu, it.aux, P), X, __shfl_sync(0xffffffffu, tk, P), __shfl_sync(0xffffffffu, nb, P));
                    }
                }
            }
            node_close(N, bm);
            if (next_lead != 0xFFFFFFFFu) {
                if (n_done == MAX_SETS) { if (lane == 0) atomicExch(&A.ctr->error, 3u); break; }
                if (lane == 0) { done[n_done][0] = M0; done[n_done][1] = M1; }
                __syncwarp();
                ++n_done;
            }
            lead = next_lead;
        }
      }
    }
    warp_epilogue(A, W, n_fresh);
}

// ---- dispatch + thread kernel.  One thread per run: buy-only runs of at most TINY_ITEMS records of a single card
// set (most runs: card sets that only pruned states ever reach) are finished right here -- the records of a run
// are in arrival order (stable sort of records generated in (parent, ordinal) order), so the first occurrence of
// a gem hand wins; every other run is appended to the list of its class (warp kernel up to BIG_W candidates, CTA
// kernel beyond: one warp on a heavy run would keep the whole grid waiting).
constexpr int TINY_ITEMS = 16;
#ifndef SPL_BIG_W
#define SPL_BIG_W 1024
#endif
constexpr uint32_t BIG_W = SPL_BIG_W;
template <bool UNORDERED>
__global__ void __launch_bounds__(TILE) m2_group_tiny_kernel(GroupArgs A, uint32_t n_runs) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint64_t s_base;
    __shared__ SmemTabs tabs;  // the buys are rebuilt from their parents (one GPU)
    if (!UNORDERED) {
        load_tabs(tabs, A.tabs);
        __syncthreads();
    }
    const unsigned lane = threadIdx.x & 31;
    const uint32_t r = blockIdx.x * TILE + threadIdx.x;
    int cls = -1;  // -1 none, 0 handled here, CLS_WARP / CLS_CTA queued
    uint32_t s = 0, cnt = 0, winmask = 0;
    uint64_t *N = nullptr;
    uint32_t n_fresh = 0;
    uint64_t kmin = ~0ull, kmax = 0;
    if (r < n_runs) {
        s = A.run_start[r];
        cnt = A.run_start[r + 1] - s;
        const uint32_t id0 = item_id(A, s);
        const uint32_t wgt = A.run_wpre[r + 1] - A.run_wpre[r];
        if (cnt <= TINY_ITEMS && id0 >= A.np) cls = 0;
        else cls = wgt <= A.warp_max ? CLS_WARP : CLS_CTA;
        if (cls == 0) {
            uint64_t lo0, hi0, M0, M1;
            load_buy_key<UNORDERED>(A, tabs, id0, lo0, hi0);
            mask_words(lo0, hi0, M0, M1);
            uint32_t gp[TINY_ITEMS / 2];  // gem hands, two per word
#pragma unroll
            for (int q = 0; q < TINY_ITEMS / 2; ++q) gp[q] = 0;
            gp[0] = (uint32_t)(lo0 & GEM_MASK);
            bool same = true;
#pragma unroll
            for (int j = 1; j < TINY_ITEMS; ++j) {
                if (j < (int)cnt) {
                    uint64_t lo, hi, m0, m1;
                    load_buy_key<UNORDERED>(A, tabs, item_id(A, s + j), lo, hi);
                    mask_words(lo, hi, m0, m1);
                    same = same && m0 == M0 && m1 == M1;
                    gp[j >> 1] |= (uint32_t)(lo & GEM_MASK) << (16 * (j & 1));
                }
            }
            if (!same) {
                cls = CLS_WARP;  // several card sets under one sort key: the warp kernel sorts that out
            } else {
                bool fresh;
                const uint64_t node = node_find_or_create(A.nodes, A.nn, M0, M1, fresh, &A.ctr->error);
                n_fresh = fresh;
                N = A.nodes + node * NODE_WORDS;
#pragma unroll
                for (int j = 0; j < TINY_ITEMS; ++j) {
                    if (j < (int)cnt) {
                        const uint32_t g = (gp[j >> 1] >> (16 * (j & 1))) & 0x7fffu;
                        bool dup = false;
                        if (!UNORDERED) {  // records in arrival order: an earlier record with the same gems wins
#pragma unroll
                            for (int i = 0; i < j; ++i) dup = dup || ((gp[i >> 1] >> (16 * (i & 1))) & 0x7fffu) == g;
                        } else {             // any order: the record with the smaller arrival index wins
                            uint32_t eq = 0;  // the other records with this gem hand (rare): compare arrival indices
#pragma unroll
                            for (int i = 0; i < TINY_ITEMS; ++i)
                                if (i != j && i < (int)cnt && ((gp[i >> 1] >> (16 * (i & 1))) & 0x7fffu) == g) eq |= 1u << i;
                            for (; eq && !dup; eq &= eq - 1)
                                dup = A.brec[item_id(A, s + (__ffs(eq) - 1)) - A.np].link < A.brec[item_id(A, s + j) - A.np].link;
                        }
                        if (!dup && (fresh || !node_bit(N, __ldg(A.gemrank + g)))) winmask |= 1u << j;
                    }
                }
            }
        }
    }
    // queue the runs of the other classes (one atomic per warp and class)
#pragma unroll
    for (int k = CLS_WARP; k <= CLS_CTA; ++k) {
        const unsigned m = __ballot_sync(0xffffffffu, cls == k);
        if (m) {
            uint32_t base = 0;
            if (lane == (unsigned)(__ffs(m) - 1)) base = atomicAdd(&A.ctr->n_cls[k], (unsigned)__popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            if (cls == k) A.cls_list[k][base + __popc(m & ((1u << lane) - 1))] = r;
        }
    }
    // winners of the runs finished here: one output reservation per CTA
    uint32_t tot;
    const uint32_t ex = block_excl_scan(__popc(winmask), warp_sums, tot);
    if (threadIdx.x == 0 && tot) s_base = A.out_base + atomicAdd(&A.ctr->n_emitted, (unsigned long long)tot);
    __syncthreads();
    uint64_t pos = s_base + ex;
    for (uint32_t m = winmask; m; m &= m - 1) {
        const int j = __ffs(m) - 1;
        Rec it;
        load_buy<UNORDERED>(A, tabs, item_id(A, s + j), it);
        st_rec(A.out + pos, it);
        const uint64_t k = flip_f64((uint64_t)__double_as_longlong(score_state(A.h, A.noise_mode, it.lo, it.hi & HI_KEY_MASK, it.aux, A.L)));
        A.out_sk[pos] = k;
        kmin = min(kmin, k); kmax = max(kmax, k);
        const uint32_t rk = __ldg(A.gemrank + (uint32_t)(it.lo & GEM_MASK));
        atomicOr(reinterpret_cast<unsigned long long *>(N + 2 + (rk >> 6)), 1ull << (rk & 63));
        ++pos;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        n_fresh += __shfl_xor_sync(0xffffffffu, n_fresh, d);
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
    }
    if (lane == 0 && n_fresh) atomicAdd(&A.ctr->n_new_nodes, n_fresh);
    if (lane == 0 && kmin <= kmax) {
        atomicMin(&A.ctr->sk_min, (unsigned long long)kmin);
        atomicMax(&A.ctr->sk_max, (unsigned long long)kmax);
    }
}

// ---- CTA kernel: runs with many items / candidates.  Direct table: min arrival index per gem hand.
struct BigSmem {
    SmemTabs tabs;
    uint64_t tbl[GEM_STATES + 6];
    uint64_t bm[NODE_BM_WORDS];
    uint64_t done0[BIG_DONE], done1[BIG_DONE];
    uint32_t warp_sums[TILE / 32 + 1];
    uint32_t job, next, fresh, n_done;
    uint64_t node, base, m0, m1;
};

// enumerate the candidates of the items of run [s, e) whose card set is (M0, M1): f(rank, t, item offset in the run)
// (spreading the takes of a batch of items evenly over the threads was measured: slower, the extra barriers cost more
// than the serial take loops)
template <bool UNORDERED, class F>
__device__ __forceinline__ void big_enumerate(const GroupArgs &A, BigSmem &S, uint32_t s, uint32_t e, uint64_t M0, uint64_t M1, F &&f) {
    for (uint32_t i = s + threadIdx.x; i < e; i += TILE) {
        const uint32_t id = item_id(A, i);
        Rec it;
        const bool isP = id < A.np;
        if (isP) ld_rec(A.front + id, it); else load_buy<UNORDERED>(A, S.tabs, id, it);
        uint64_t m0, m1;
        mask_words(it.lo, it.hi, m0, m1);
        if (m0 != M0 || m1 != M1) {  // another card set with the same sort key: remember the first one not done yet
            bool done = false;
            for (uint32_t d = 0; d < S.n_done; ++d) done |= (S.done0[d] == m0 && S.done1[d] == m1);
            if (!done) atomicMin(&S.next, i);
            continue;
        }
        if (!isP) {
            f((uint32_t)__ldg(A.gemrank + (uint32_t)(it.lo & GEM_MASK)), it.link, i - s);
        } else {
            uint64_t bl, bh;
            uint32_t nb, tk;
            derive_parent(S.tabs, A.takes_idx, it.lo, it.hi, it.aux, bl, bh, nb, tk);
            const uint64_t tb = (parent_rank(A, id) << 8) | nb;
            const uint32_t ntk = tk & 0xff;
            for (uint32_t q = 0; q < ntk; ++q) f((uint32_t)__ldg(A.gemrank + __ldg(A.takes_edges + (tk >> 8) + q)), tb + q, i - s);
        }
    }
}

template <bool UNORDERED>
__global__ void __launch_bounds__(TILE) m2_group_big_kernel(GroupArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BigSmem &S = *reinterpret_cast<BigSmem *>(smem_raw);
    const unsigned tid = threadIdx.x, lane = tid & 31;
    load_tabs(S.tabs, A.tabs);
    const uint32_t n_big = A.ctr->n_cls[CLS_CTA];
    uint32_t n_fresh = 0;
    uint64_t kmin = ~0ull, kmax = 0;
    uint32_t ticket = 0;  // (thread 0) the next job, fetched while the current one is processed
    if (tid == 0) ticket = atomicAdd(&A.ctr->ticket[3], 1u);
    for (;;) {
        __syncthreads();
        if (tid == 0) {
            S.job = ticket;
            if (ticket < n_big) ticket = atomicAdd(&A.ctr->ticket[3], 1u);
        }
        __syncthreads();
        if (S.job >= n_big) break;
        const uint32_t r = A.cls_list[CLS_CTA][S.job];
        const uint32_t s = A.run_start[r], e = A.run_start[r + 1];
        if (tid == 0) { S.n_done = 0; S.next = s; }
        __syncthreads();
        while (S.next != 0xFFFFFFFFu) {  // one iteration per distinct card set of the run
            const uint32_t lead = S.next;
            __syncthreads();
            if (tid == 0) {
                const uint32_t id = item_id(A, lead);
                Rec src;
                if (id < A.np) ld_rec(A.front + id, src); else load_buy<UNORDERED>(A, S.tabs, id, src);
                mask_words(src.lo, src.hi, S.m0, S.m1);
                bool fresh;
                S.node = node_find_or_create(A.nodes, A.nn, S.m0, S.m1, fresh, &A.ctr->error);
                S.fresh = fresh;
                n_fresh += fresh;
                S.next = 0xFFFFFFFFu;
            }
            __syncthreads();
            const uint64_t M0 = S.m0, M1 = S.m1;
            uint64_t *N = A.nodes + S.node * NODE_WORDS;
            for (int i = tid; i < GEM_STATES; i += TILE) S.tbl[i] = ~0ull;
            if (tid < NODE_BM_WORDS) S.bm[tid] = S.fresh ? 0ull : N[2 + tid];
            __syncthreads();
            // pass 0: first arrival per gem hand among the candidates not in the visited set; the table word is
            // arrival index << 24 | offset of the producing item in the run (a run holds < 2^24 items: at most
            // BIG_DONE + 1 card sets of <= 2898 parents and their predecessors' buy records; arrival indices are < 2^40)
            big_enumerate<UNORDERED>(A, S, s, e, M0, M1, [&](uint32_t rk, uint64_t t, uint32_t at) {
                if (!((S.bm[rk >> 6] >> (rk & 63)) & 1))
                    atomicMin(reinterpret_cast<unsigned long long *>(&S.tbl[rk]), (unsigned long long)((t << BIG_AT_BITS) | at));
            });
            __syncthreads();
            // pass 1: the occupied table entries are the winners; each is rebuilt from its producing item
            uint32_t mywins = 0;
            for (uint32_t rk = tid; rk < GEM_STATES; rk += TILE) mywins += S.tbl[rk] != ~0ull;
            uint32_t tot;
            const uint32_t ex = block_excl_scan(mywins, S.warp_sums, tot);
            if (tid == 0) S.base = A.out_base + atomicAdd(&A.ctr->n_emitted, (unsigned long long)tot);
            __syncthreads();
            uint64_t pos = S.base + ex;
            for (uint32_t rk = tid; rk < GEM_STATES; rk += TILE) {
                const uint64_t v = S.tbl[rk];
                if (v == ~0ull) continue;
                const uint32_t id = item_id(A, s + (uint32_t)(v & ((1u << BIG_AT_BITS) - 1)));
                Rec o;
                if (id < A.np) {  // a gem take of that parent: same cards, saved, points and bonus
                    ld_rec(A.front + id, o);
                    o.lo = (o.lo & ~GEM_MASK) | __ldg(A.rankgems + rk);
                } else {
                    load_buy<UNORDERED>(A, S.tabs, id, o);
                }
                o.link = v >> BIG_AT_BITS;
                st_rec(A.out + pos, o);
                if (A.out_sk) {
                    const uint64_t k = flip_f64((uint64_t)__double_as_longlong(score_state(A.h, A.noise_mode, o.lo, o.hi & HI_KEY_MASK, o.aux, A.L)));
                    A.out_sk[pos] = k;
                    kmin = min(kmin, k); kmax = max(kmax, k);
                }
                ++pos;
                atomicOr(reinterpret_cast<unsigned *>(S.bm) + (rk >> 5), 1u << (rk & 31));
            }
            __syncthreads();
            if (tid < NODE_BM_WORDS) N[2 + tid] = S.bm[tid];
            if (tid == 0) {
                if (S.n_done < BIG_DONE) { S.done0[S.n_done] = M0; S.done1[S.n_done] = M1; ++S.n_done; }
                else if (S.next != 0xFFFFFFFFu) { atomicExch(&A.ctr->error, 3u); S.next = 0xFFFFFFFFu; }
            }
            __syncthreads();
        }
    }
    if (tid == 0 && n_fresh) atomicAdd(&A.ctr->n_new_nodes, n_fresh);
    if (A.out_sk) {
#pragma unroll
        for (int d = 16; d; d >>= 1) {
            kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
            kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
        }
        if (lane == 0 && kmin <= kmax) {
            atomicMin(&A.ctr->sk_min, (unsigned long long)kmin);
            atomicMax(&A.ctr->sk_max, (unsigned long long)kmax);
        }
    }
}

}  // namespace spl
