// spl_realistic.cuh -- realistic multi-player mode (reference: src/solver.py:25-200, 471-860).
//
// State record RRec (96 B = three 32-byte sectors):
//   p[4]    per player: 90-bit card mask (mlo: cards 0..63, mhi: 64..89), gems (3 bits/colour), saved
//   vis[12] visible card per market slot, tier-major, in slot order (255 = empty, empties trail)
//   cur     current player;   link = parent_rank << 8 | ordinal
// Everything else the reference keeps in MultiPlayerState is derived on the fly:
//   bonus[c] / pts  : popcounts of the card mask against colour / point masks
//   gem pool        : gems_per_color - sum of the players' gems (conservation, :600-604, :685)
//   deck position   : 4 + #cards of the tier owned by anyone            (CardMarket.buy_card :121-170)
//   is_game_over()  : players[cur].pts >= target  (final round ends when play returns to its trigger, :542-549)
// Identity (src/solver.py:495-500) = (players incl. saved, pool, visible cards in slot order, current
// player).  The visited set is keyed by an EXACT 384-bit packing of those fields (r_pack_key): card owner codes,
// gems and saved per player, the deck position of every visible slot, the current player; the pool is a function
// of the players' gems.  (The reference itself dedups on a 64-bit hash of the same fields.)
#pragma once
#include "spl_kernels.cuh"

namespace spl {

struct RPlayer {
    uint64_t mlo;
    uint32_t mhi;
    uint16_t gems, saved;
};
struct __align__(32) RRec {
    RPlayer p[4];
    uint8_t vis[12];
    uint8_t cur, pad[3];
    uint64_t link, spare;
};
static_assert(sizeof(RRec) == 96, "RRec layout");

struct RConfigDev {
    int32_t P, target, gpc, noise;
    int32_t deck_len[3];
    uint8_t deck[3][40];
    uint64_t col_lo[NCOL], pt_lo[6], tier_lo[3];
    uint32_t col_hi[NCOL], pt_hi[6], tier_hi[3];
    uint32_t card[SPL_NUM_CARDS];
    uint8_t pos_of[SPL_NUM_CARDS];  // position of a card inside its tier's deck sequence
};

// the RRec overloads of ld_rec / st_rec (spl_common.cuh): three 32-byte sectors
__device__ __forceinline__ void ld_rec(const RRec *p, RRec &r) {
    const ulonglong4 *s = reinterpret_cast<const ulonglong4 *>(p);
    ulonglong4 *d = reinterpret_cast<ulonglong4 *>(&r);
    d[0] = s[0]; d[1] = s[1]; d[2] = s[2];
}
__device__ __forceinline__ void st_rec(RRec *p, const RRec &r) {
    const ulonglong4 *s = reinterpret_cast<const ulonglong4 *>(&r);
    ulonglong4 *d = reinterpret_cast<ulonglong4 *>(p);
    d[0] = s[0]; d[1] = s[1]; d[2] = s[2];
}

__device__ __forceinline__ void r_derive(const RConfigDev &C, const RPlayer &p, int bonus[NCOL], int &pts) {
#pragma unroll
    for (int c = 0; c < NCOL; ++c) bonus[c] = __popcll(p.mlo & C.col_lo[c]) + __popc(p.mhi & C.col_hi[c]);
    pts = 0;
#pragma unroll
    for (int v = 1; v <= 5; ++v) pts += v * (__popcll(p.mlo & C.pt_lo[v]) + __popc(p.mhi & C.pt_hi[v]));
}
__device__ __forceinline__ int r_pts(const RConfigDev &C, const RPlayer &p) {
    int pts = 0;
#pragma unroll
    for (int v = 1; v <= 5; ++v) pts += v * (__popcll(p.mlo & C.pt_lo[v]) + __popc(p.mhi & C.pt_hi[v]));
    return pts;
}
// PlayerState.can_afford (src/solver.py:192-200): gems + bonus >= cost per colour, no clamp
__device__ __forceinline__ bool r_can_afford(const RConfigDev &C, uint32_t gems, const int bonus[NCOL], int card) {
    const uint32_t cd = C.card[card];
    bool ok = true;
#pragma unroll
    for (int c = 0; c < NCOL; ++c) ok &= (int)((gems >> (3 * c)) & 7) + bonus[c] >= (int)((cd >> (3 * c)) & 7);
    return ok;
}

// 27 successor slots in the reference's order (:573-748): 12 buys in market slot order, the 10
// colour triples in combinations() order, the 5 double takes.  Returns the valid-slot mask.
__device__ __forceinline__ uint32_t r_valid_mask(const RConfigDev &C, const RRec &s, const int bonus[NCOL]) {
    const RPlayer &me = s.p[s.cur];
    int pool[NCOL], hand = 0;
#pragma unroll
    for (int c = 0; c < NCOL; ++c) {
        int tot = 0;
        for (int q = 0; q < C.P; ++q) tot += (s.p[q].gems >> (3 * c)) & 7;
        pool[c] = C.gpc - tot;
        hand += (me.gems >> (3 * c)) & 7;
    }
    uint32_t m = 0;
    for (int k = 0; k < 12; ++k)
        if (s.vis[k] != 255 && r_can_afford(C, me.gems, bonus, s.vis[k])) m |= 1u << k;
    if (hand + 3 <= 10) {
        int k = 12;
        for (int a = 0; a < NCOL; ++a)
            for (int b = a + 1; b < NCOL; ++b)
                for (int c = b + 1; c < NCOL; ++c, ++k)
                    if (pool[a] > 0 && pool[b] > 0 && pool[c] > 0) m |= 1u << k;
    }
    if (hand + 2 <= 10)
        for (int c = 0; c < NCOL; ++c)
            if (pool[c] >= 4) m |= 1u << (22 + c);
    return m;
}

__device__ __forceinline__ void r_make_child(const RConfigDev &C, const RRec &s, const int bonus[NCOL], int slot, RRec &o) {
    o = s;
    const int cur = s.cur;
    RPlayer &me = o.p[cur];
    o.cur = (uint8_t)((cur + 1) % C.P);
    if (slot < 12) {  // buy (:574-632)
        const int card = s.vis[slot];
        const uint32_t cd = C.card[card];
        uint32_t ng = 0, saved = 0;
#pragma unroll
        for (int c = 0; c < NCOL; ++c) {
            const int cost = (cd >> (3 * c)) & 7;
            const int pay = max(cost - bonus[c], 0);
            saved += cost - pay;
            ng |= (uint32_t)max((int)((me.gems >> (3 * c)) & 7) - pay, 0) << (3 * c);
        }
        me.gems = (uint16_t)ng;
        me.saved = (uint16_t)(me.saved + saved);
        if (card < 64) me.mlo |= 1ull << card; else me.mhi |= 1u << (card - 64);
        const int t = slot >> 2;
        int bought = 0;
        for (int q = 0; q < C.P; ++q) bought += __popcll(s.p[q].mlo & C.tier_lo[t]) + __popc(s.p[q].mhi & C.tier_hi[t]);
        const int pos = 4 + bought;
        for (int k = slot & 3; k < 3; ++k) o.vis[t * 4 + k] = s.vis[t * 4 + k + 1];
        o.vis[t * 4 + 3] = 255;
        if (pos < C.deck_len[t]) {
            int e = 0;
            while (e < 4 && o.vis[t * 4 + e] != 255) ++e;
            o.vis[t * 4 + e] = C.deck[t][pos];
        }
    } else if (slot < 22) {  // three different colours (:671-707)
        int k = 12;
        for (int a = 0; a < NCOL; ++a)
            for (int b = a + 1; b < NCOL; ++b)
                for (int c = b + 1; c < NCOL; ++c, ++k)
                    if (k == slot) me.gems = (uint16_t)(me.gems + (1 << (3 * a)) + (1 << (3 * b)) + (1 << (3 * c)));
    } else {  // two of one colour (:710-748)
        me.gems = (uint16_t)(me.gems + (2 << (3 * (slot - 22))));
    }
}

// ------------------------------------------------------------------ exact identity key (384 bits)
// Injective packing of MultiPlayerState's identity (src/solver.py:495-500; PlayerState :177-186):
//   owner of every card : 2 bits x 90 (0 = nobody, 1 + player) for 2-3 players; three cards per 7 bits (base 5)
//                         for 4 players                                                   180 | 210 bits
//   per player          : gems 15 bits, saved 10 bits                                     25 x P
//   market              : deck position (6 bits, 63 = empty) of each of the 12 slots, in slot order   72 bits
//   current player      : 2 bits
// = 304 / 329 / 384 bits for 2 / 3 / 4 players.  bonus and pts are functions of the cards, the pool of the gems.
constexpr int RKEY_WORDS = 6;
struct RKeyWriter {
    uint64_t w[RKEY_WORDS];
    int at;
    __device__ __forceinline__ void put(uint64_t v, int bits) {
        const int i = at >> 6, o = at & 63;
        w[i] |= v << o;
        if (o + bits > 64) w[i + 1] |= v >> (64 - o);
        at += bits;
    }
};
// returns false if a field does not fit (saved >= 1024): the caller raises an error instead of merging states
__device__ __forceinline__ bool r_pack_key(const RConfigDev &C, const RRec &s, uint64_t key[RKEY_WORDS]) {
    RKeyWriter K;
#pragma unroll
    for (int i = 0; i < RKEY_WORDS; ++i) K.w[i] = 0;
    K.at = 0;
    bool ok = true;
    auto owner = [&](int card) -> uint32_t {
        for (int q = 0; q < C.P; ++q)
            if (card < 64 ? (s.p[q].mlo >> card) & 1 : (s.p[q].mhi >> (card - 64)) & 1) return (uint32_t)q + 1;
        return 0u;
    };
    if (C.P <= 3) {
        for (int card = 0; card < SPL_NUM_CARDS; ++card) K.put(owner(card), 2);
    } else {
        for (int card = 0; card < SPL_NUM_CARDS; card += 3) K.put(owner(card) + 5 * owner(card + 1) + 25 * owner(card + 2), 7);
    }
    for (int q = 0; q < C.P; ++q) {
        K.put(s.p[q].gems & 0x7fffu, 15);
        ok &= s.p[q].saved < 1024;
        K.put(s.p[q].saved & 1023u, 10);
    }
    for (int k = 0; k < 12; ++k) K.put(s.vis[k] == 255 ? 63u : (uint32_t)C.pos_of[s.vis[k]], 6);
    K.put(s.cur, 2);
#pragma unroll
    for (int i = 0; i < RKEY_WORDS; ++i) key[i] = K.w[i];
    return ok;
}
__device__ __forceinline__ uint64_t r_key_hash(const uint64_t key[RKEY_WORDS]) {
    uint64_t h = 0x243F6A8885A308D3ull;
#pragma unroll
    for (int i = 0; i < RKEY_WORDS; i += 2) h = mix64(h ^ key[i], key[i + 1] + 0x9E3779B97F4A7C15ull * (uint64_t)(i + 1));
    return h;
}

// Visited table of realistic mode: 64-byte buckets, one state each: {key[6], ctrl, ~t, pad}.
//   ctrl = 0 empty | tag << 8 | 1 claimed, key being written | tag << 8 | 3 ready.  tag = epoch (level) of insertion.
// A bucket is claimed with one 64-bit CAS on ctrl; the claimer writes the key and publishes ctrl = ready.  A probe that
// meets a claimed bucket waits for the key (the writer is running and waits for nobody), then compares all 384 bits.
// ~t (t = arrival index in the epoch): atomicMax keeps the FIRST arrival, as in the speedrun table.
struct __align__(64) RBucket {
    uint64_t key[RKEY_WORDS];
    unsigned long long ctrl;
    unsigned int tinv, pad;
};
static_assert(sizeof(RBucket) == 64, "RBucket layout");
constexpr uint32_t R_DEAD = 0xFFFFFFFFu;

__device__ __forceinline__ uint32_t r_probe(RBucket *__restrict__ table, uint64_t nb, uint64_t tag, const uint64_t key[RKEY_WORDS],
                                            uint32_t tinv, uint32_t &n_new, unsigned int *error) {
    uint64_t b = __umul64hi(r_key_hash(key), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        RBucket *B = table + b;
        unsigned long long c = *reinterpret_cast<volatile unsigned long long *>(&B->ctrl);
        if (c == 0) {
            c = atomicCAS(&B->ctrl, 0ull, (unsigned long long)(tag << 8 | 1));
            if (c == 0) {  // claimed: write the key, then publish
#pragma unroll
                for (int i = 0; i < RKEY_WORDS; ++i) B->key[i] = key[i];
                __threadfence();
                atomicExch(&B->ctrl, (unsigned long long)(tag << 8 | 3));
                ++n_new;
                atomicMax(&B->tinv, tinv);
                return (uint32_t)b;
            }
        }
        while ((c & 3) == 1) c = *reinterpret_cast<volatile unsigned long long *>(&B->ctrl);  // key not published yet
        __threadfence();
        bool same = true;
#pragma unroll
        for (int i = 0; i < RKEY_WORDS; ++i) same &= *reinterpret_cast<volatile uint64_t *>(&B->key[i]) == key[i];
        if (same) {
            if ((c >> 8) != tag) return R_DEAD;  // visited in an earlier level
            if (*reinterpret_cast<volatile unsigned int *>(&B->tinv) > tinv) return R_DEAD;  // an earlier arrival is registered
            atomicMax(&B->tinv, tinv);
            return (uint32_t)b;
        }
        if (++b == nb) b = 0;
    }
    atomicExch(error, 1u);
    return R_DEAD;
}

// exact-key probe / insert of a materialised successor list (arrival index = list index)
__global__ void __launch_bounds__(TILE) r_probe_kernel(const RRec *__restrict__ cand, int64_t n, const RConfigDev *__restrict__ cfg,
                                                       RBucket *__restrict__ table, uint64_t nb, uint64_t tag,
                                                       uint32_t *__restrict__ cand_slot, Counters *ctr) {
    const int64_t t = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint32_t n_new = 0;
    if (t < n) {
        RRec s;
        ld_rec(cand + t, s);
        uint64_t key[RKEY_WORDS];
        if (!r_pack_key(*cfg, s, key)) atomicExch(&ctr->error, 4u);
        cand_slot[t] = r_probe(table, nb, tag, key, ~(uint32_t)t, n_new, &ctr->error);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
    if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(&ctr->n_new, (unsigned long long)n_new);
}
// winners (first arrivals of new states) in arrival order: out_idx[rank] = list index; 8 candidates per thread
__global__ void __launch_bounds__(TILE) r_winners_kernel(const uint32_t *__restrict__ cand_slot, const RBucket *__restrict__ table,
                                                         int64_t n, int64_t *__restrict__ out_idx, uint64_t *status, Counters *ctr,
                                                         int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * 8;
    uint32_t mask = 0;
    for (int q = 0; q < 8; ++q)
        if (b0 + q < n) {
            const uint32_t sl = cand_slot[b0 + q];
            if (sl != R_DEAD && ~ld_cg_u32(&table[sl].tinv) == (uint32_t)(b0 + q)) mask |= 1u << q;
        }
    uint32_t tot;
    const uint32_t ex = block_excl_scan(__popc(mask), warp_sums, tot);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, tot, 0);
        if (threadIdx.x == 0) {
            s_base = e;
            if (((int64_t)tile + 1) * TILE * 8 >= n) ctr->n_emitted = e + tot;
        }
    }
    __syncthreads();
    uint64_t pos = s_base + ex;
    for (; mask; mask &= mask - 1) out_idx[pos++] = b0 + (__ffs(mask) - 1);
}
// move every ready bucket of an old table into a larger one (tags preserved)
__global__ void __launch_bounds__(TILE) r_rehash_kernel(const RBucket *__restrict__ old_table, uint64_t old_nb,
                                                        RBucket *__restrict__ table, uint64_t nb, Counters *ctr) {
    const uint64_t i = (uint64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= old_nb || old_table[i].ctrl == 0) return;
    uint64_t key[RKEY_WORDS];
#pragma unroll
    for (int k = 0; k < RKEY_WORDS; ++k) key[k] = old_table[i].key[k];
    uint64_t b = __umul64hi(r_key_hash(key), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        if (atomicCAS(&table[b].ctrl, 0ull, old_table[i].ctrl) == 0) {
#pragma unroll
            for (int k = 0; k < RKEY_WORDS; ++k) table[b].key[k] = key[k];
            return;
        }
        if (++b == nb) b = 0;
    }
    atomicExch(&ctr->error, 1u);
}
// the packed keys of a batch (tests: injectivity against the identity bytes)
__global__ void __launch_bounds__(TILE) r_pack_kernel(const RRec *__restrict__ recs, int64_t n, const RConfigDev *__restrict__ cfg,
                                                      uint64_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    RRec s;
    ld_rec(recs + i, s);
    uint64_t key[RKEY_WORDS];
    r_pack_key(*cfg, s, key);
#pragma unroll
    for (int k = 0; k < RKEY_WORDS; ++k) out[i * RKEY_WORDS + k] = key[k];
}

// multi_competitive_heuristic (src/solver.py:778-812), bit-exact: LUT pows, separately rounded ops
__device__ __forceinline__ double r_score(const RConfigDev &C, const RRec &s, const ScoreLuts &L, int r_ext = 50) {
    const int prev = (s.cur + C.P - 1) % C.P;
    const RPlayer &me = s.p[prev], &opp = s.p[s.cur];
    int bm[NCOL], bo[NCOL], pm, po, rm = 0, ro = 0, nnz = 0, am = 0, ao = 0;
    r_derive(C, me, bm, pm);
    r_derive(C, opp, bo, po);
#pragma unroll
    for (int c = 0; c < NCOL; ++c) {
        rm += ((me.gems >> (3 * c)) & 7) + 2 * bm[c];
        ro += ((opp.gems >> (3 * c)) & 7) + 2 * bo[c];
        nnz += bm[c] > 0;
    }
    for (int k = 0; k < 12; ++k)
        if (s.vis[k] != 255) {
            am += r_can_afford(C, me.gems, bm, s.vis[k]);
            ao += r_can_afford(C, opp.gems, bo, s.vis[k]);
        }
    // point_diff = d**2.5 if me.pts > opp.pts else -(d**2.5)   (-0.0 when equal)
    const double pw = __ldg(L.pts + 0 * 256 + abs(pm - po));
    const double pd = pm > po ? pw : -pw;
    double acc = __dmul_rn(pd, 100.0);
    // resource_diff * 20: float when positive, the int 0 otherwise (x + 0 == x + 0.0)
    acc = __dadd_rn(acc, rm > ro ? __dmul_rn(__ldg(L.small + 3 * 512 + (rm - ro)), 20.0) : 0.0);
    acc = __dadd_rn(acc, (double)((am - ao) * 5));
    acc = __dadd_rn(acc, __dmul_rn(__ldg(L.small + 3 * 512 + nnz), 3.0));
    int r = C.noise == 2 ? r_ext : 50;
    if (C.noise == 1) {
        uint64_t h = 0;
        for (int q = 0; q < C.P; ++q)
            h = mix64(h ^ s.p[q].mlo, (uint64_t)s.p[q].mhi | (uint64_t)s.p[q].gems << 32 | (uint64_t)s.p[q].saved << 48);
        r = 1 + (int)(h % 100ull);
    }
    return __dadd_rn(acc, __dmul_rn((double)r, 0.01));
}

// ------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(TILE) r_goal_kernel(const RRec *__restrict__ front, int64_t n,
                                                      const RConfigDev *__restrict__ cfg, Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    long long r = 0x7fffffffffffffffll;
    if (i < n) {
        const RPlayer p = front[i].p[front[i].cur];
        if (r_pts(*cfg, p) >= cfg->target) r = i;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) r = min(r, __shfl_xor_sync(0xffffffffu, r, d));
    if ((threadIdx.x & 31) == 0 && r != 0x7fffffffffffffffll) atomicMin(&ctr->goal_rank, r);
}

__global__ void __launch_bounds__(TILE) r_count_scan_kernel(const RRec *__restrict__ front, int64_t n,
                                                            const RConfigDev *__restrict__ cfg, uint32_t *__restrict__ off,
                                                            uint32_t *__restrict__ vmask, uint64_t *status, Counters *ctr,
                                                            int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t p = (int64_t)tile * TILE + threadIdx.x;
    uint32_t cnt = 0, m = 0;
    if (p < n) {
        RRec s;
        ld_rec(front + p, s);
        int bonus[NCOL], pts;
        r_derive(*cfg, s.p[s.cur], bonus, pts);
        m = r_valid_mask(*cfg, s, bonus);
        cnt = __popc(m);
        vmask[p] = m;
    }
    uint32_t total;
    const uint32_t excl = block_excl_scan(cnt, warp_sums, total);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, total, 0);
        if (threadIdx.x == 0) {
            s_base = e;
            if ((int64_t)(tile + 1) * TILE >= n) ctr->total_cands = e + total;
        }
    }
    __syncthreads();
    if (p < n) off[p] = (uint32_t)(s_base + excl);
}

// one thread per parent: write its successors at off[parent] + ordinal
__global__ void __launch_bounds__(TILE) r_expand_kernel(const RRec *__restrict__ front, int64_t n,
                                                        const RConfigDev *__restrict__ cfg,
                                                        const uint32_t *__restrict__ off,
                                                        const uint32_t *__restrict__ vmask, int64_t rank_base,
                                                        RRec *__restrict__ cand) {
    const int64_t p = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (p >= n) return;
    RRec s;
    ld_rec(front + p, s);
    int bonus[NCOL], pts;
    r_derive(*cfg, s.p[s.cur], bonus, pts);
    uint32_t m = vmask[p], ord = 0;
    uint64_t t = off[p];
    while (m) {
        const int slot = __ffs(m) - 1;
        m &= m - 1;
        RRec o;
        r_make_child(*cfg, s, bonus, slot, o);
        o.link = ((uint64_t)(rank_base + p) << 8) | ord;
        o.spare = 0;
        st_rec(cand + t, o);
        ++t;
        ++ord;
    }
}

template <typename IDX>
__global__ void __launch_bounds__(TILE) r_gather_kernel(const RRec *__restrict__ src, const IDX *__restrict__ idx, int64_t n,
                                                        RRec *__restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        RRec r;
        ld_rec(src + idx[i], r);
        st_rec(dst + i, r);
    }
}

__global__ void __launch_bounds__(TILE) r_score_kernel(const RRec *__restrict__ recs, int64_t n,
                                                       const RConfigDev *__restrict__ cfg, ScoreLuts L,
                                                       uint64_t *__restrict__ sk, double *__restrict__ raw, Counters *ctr,
                                                       const uint8_t *__restrict__ draws = nullptr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint64_t kmin = ~0ull, kmax = 0;
    if (i < n) {
        RRec s;
        ld_rec(recs + i, s);
        const double sc = r_score(*cfg, s, L, draws ? draws[i] : 50);
        if (raw) raw[i] = sc;
        if (sk) {
            const uint64_t k = flip_f64((uint64_t)__double_as_longlong(sc));
            sk[i] = k;
            kmin = kmax = k;
        }
    }
    if (sk) {
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

// max over players of pts, per state (the reference's progress line, src/solver.py:832-836)
__global__ void __launch_bounds__(TILE) r_maxpts_kernel(const RRec *__restrict__ recs, int64_t n,
                                                        const RConfigDev *__restrict__ cfg, uint8_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        int m = 0;
        for (int q = 0; q < cfg->P; ++q) m = max(m, r_pts(*cfg, recs[i].p[q]));
        out[i] = (uint8_t)min(m, 255);
    }
}

__global__ void __launch_bounds__(TILE) r_links_kernel(const RRec *__restrict__ recs, int64_t n, uint64_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) out[i] = recs[i].link;
}

// ------------------------------------------------------------------ key-sharded driver (sharded.py: RCudaBackend)
// Owner rank of a state: the LOW 32 bits of r_key_hash, mapped onto [0, n_ranks) by a multiply-shift.  The owner's
// table takes the bucket from the HIGH bits (__umul64hi(hash, nb) with nb < 2^32 buckets), so which rank owns a state
// says nothing about its bucket there, and every owner fills its whole table evenly.
__device__ __forceinline__ uint32_t r_owner_of(uint64_t h, uint32_t n_ranks) {
    return (uint32_t)(((h & 0xffffffffull) * n_ranks) >> 32);
}
// packed key + owner (sort digit) + identity permutation of every candidate
__global__ void __launch_bounds__(TILE) r_route_pack_kernel(const RRec *__restrict__ cand, int64_t n, const RConfigDev *__restrict__ cfg,
                                                            uint32_t n_ranks, uint64_t *__restrict__ keys, uint64_t *__restrict__ owner,
                                                            uint32_t *__restrict__ idx, Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    RRec s;
    ld_rec(cand + i, s);
    uint64_t key[RKEY_WORDS];
    if (!r_pack_key(*cfg, s, key)) atomicExch(&ctr->error, 4u);
#pragma unroll
    for (int k = 0; k < RKEY_WORDS; ++k) keys[i * RKEY_WORDS + k] = key[k];
    owner[i] = r_owner_of(r_key_hash(key), n_ranks);
    idx[i] = (uint32_t)i;
}
// send buffer: the keys in (owner, arrival) order; perm keeps that order for spl_rcompact_winners
__global__ void __launch_bounds__(TILE) r_gather_keys_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ idx,
                                                             int64_t n, uint64_t *__restrict__ out, uint32_t *__restrict__ perm) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = idx[i];
#pragma unroll
    for (int k = 0; k < RKEY_WORDS; ++k) out[i * RKEY_WORDS + k] = keys[(int64_t)j * RKEY_WORDS + k];
    perm[i] = j;
}
// first-arrival insert of a list of packed keys (arrival index = list index)
__global__ void __launch_bounds__(TILE) r_probe_keys_kernel(const uint64_t *__restrict__ keys, int64_t n, RBucket *__restrict__ table,
                                                            uint64_t nb, uint64_t tag, uint32_t *__restrict__ cand_slot, Counters *ctr) {
    const int64_t t = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint32_t n_new = 0;
    if (t < n) {
        uint64_t key[RKEY_WORDS];
#pragma unroll
        for (int k = 0; k < RKEY_WORDS; ++k) key[k] = keys[t * RKEY_WORDS + k];
        cand_slot[t] = r_probe(table, nb, tag, key, ~(uint32_t)t, n_new, &ctr->error);
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
    if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(&ctr->n_new, (unsigned long long)n_new);
}
// the ~t word of a realistic bucket: the slot_tword overload win_flags_kernel reads
__device__ __forceinline__ const uint32_t *slot_tword(const RBucket *table, uint32_t sl) { return &table[sl].tinv; }

// ------------------------------------------------------------------ row layer of the key-sharded driver, for both row kinds:
// R = Rec (speedrun, 32 B) or RRec (realistic, 96 B) through the ld_rec / st_rec overloads; Table = the speedrun table's
// uint64_t words or RBucket through the slot_tword overloads (R_DEAD == DEAD)
// winner byte per listed candidate: its slot still holds its own arrival index
template <typename Table>
__global__ void __launch_bounds__(TILE) win_flags_kernel(const uint32_t *__restrict__ cand_slot, const Table *__restrict__ table,
                                                         int64_t n, uint8_t *__restrict__ flags) {
    const int64_t t = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (t < n) {
        const uint32_t s = cand_slot[t];
        flags[t] = s != DEAD && ~ld_cg_u32(slot_tword(table, s)) == (uint32_t)t;
    }
}
// stable compaction of the flagged rows (arrival order preserved): 8 rows per thread, look-back scan
template <typename R>
__global__ void __launch_bounds__(TILE) compact_rows_kernel(const R *__restrict__ rows, const uint8_t *__restrict__ flags,
                                                            int64_t n, R *__restrict__ out, uint64_t *status,
                                                            Counters *ctr, int ticket_id) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t b0 = ((int64_t)tile * TILE + threadIdx.x) * 8;
    uint32_t mask = 0;
    if (b0 + 8 <= n) {
        const uint64_t f = *reinterpret_cast<const uint64_t *>(flags + b0);
#pragma unroll
        for (int q = 0; q < 8; ++q) mask |= (uint32_t)((f >> (8 * q)) & 1) << q;
    } else {
        for (int q = 0; q < 8; ++q)
            if (b0 + q < n && flags[b0 + q]) mask |= 1u << q;
    }
    uint32_t tot;
    const uint32_t ex = block_excl_scan(__popc(mask), warp_sums, tot);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, tot, 0);
        if (threadIdx.x == 0) {
            s_base = e;
            if (((int64_t)tile + 1) * TILE * 8 >= n) ctr->n_emitted = e + tot;
        }
    }
    __syncthreads();
    uint64_t pos = s_base + ex;
    while (mask) {
        const int q = __ffs(mask) - 1;
        mask &= mask - 1;
        R r;
        ld_rec(rows + b0 + q, r);
        st_rec(out + pos, r);
        ++pos;
    }
}
// out[i] = rows[idx[i]] (gather) or out[idx[i]] = rows[i] (scatter), 64-bit indices
template <typename R>
__global__ void __launch_bounds__(TILE) move_rows_kernel(const R *__restrict__ rows, const int64_t *__restrict__ idx,
                                                         int64_t n, R *__restrict__ out, int scatter) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        R r;
        ld_rec(rows + (scatter ? i : idx[i]), r);
        st_rec(out + (scatter ? idx[i] : i), r);
    }
}

// ------------------------------------------------------------------ batched search (spl_rbatch_*): B games in lockstep
// Every per-record array of a batch level is game-major: game g owns the index range seg[g] .. seg[g + 1] (seg[0] = 0,
// seg[B] = n; a game that has ended owns an empty range), and inside it the records keep the order the single-game
// solver gives them.  Link words carry the parent's rank inside its game, so each game's segment of the queue is
// byte-identical to spl_rsolver's queue.  cfg[g] is game g's RConfigDev.
//
// The batch's visited table holds (game, exact key) entries: RBucket.pad is the game, and the game is mixed into the
// bucket hash, so that B games sharing a root (every 2-player game starts from the same key) do not share a probe run.
__device__ __forceinline__ int rb_game_of(const int64_t *__restrict__ seg, int n_games, int64_t i) {
    int lo = 0, hi = n_games;  // seg[lo] <= i < seg[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(seg + mid) <= i) lo = mid; else hi = mid;
    }
    return lo;
}
// ctr[g] += v, one atomic per run of lanes of a warp that share a game (every lane calls it; g < 0: nothing to add)
__device__ __forceinline__ void rb_warp_add(unsigned long long *ctr, int g, uint32_t v) {
    const unsigned peers = __match_any_sync(0xffffffffu, g);
    const uint32_t sum = __reduce_add_sync(peers, v);
    if (g >= 0 && sum && (int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(ctr + g, (unsigned long long)sum);
}
__device__ __forceinline__ uint64_t rb_key_hash(const uint64_t key[RKEY_WORDS], uint32_t game) {
    return mix64(r_key_hash(key), 0x9E3779B97F4A7C15ull * ((uint64_t)game + 1));
}

// r_probe with the game as part of the identity
__device__ __forceinline__ uint32_t rb_probe(RBucket *__restrict__ table, uint64_t nb, uint64_t tag, const uint64_t key[RKEY_WORDS],
                                             uint32_t game, uint32_t tinv, uint32_t &n_new, unsigned int *error) {
    uint64_t b = __umul64hi(rb_key_hash(key, game), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        RBucket *B = table + b;
        unsigned long long c = *reinterpret_cast<volatile unsigned long long *>(&B->ctrl);
        if (c == 0) {
            c = atomicCAS(&B->ctrl, 0ull, (unsigned long long)(tag << 8 | 1));
            if (c == 0) {
#pragma unroll
                for (int i = 0; i < RKEY_WORDS; ++i) B->key[i] = key[i];
                B->pad = game;
                __threadfence();
                atomicExch(&B->ctrl, (unsigned long long)(tag << 8 | 3));
                ++n_new;
                atomicMax(&B->tinv, tinv);
                return (uint32_t)b;
            }
        }
        while ((c & 3) == 1) c = *reinterpret_cast<volatile unsigned long long *>(&B->ctrl);
        __threadfence();
        bool same = *reinterpret_cast<volatile unsigned int *>(&B->pad) == game;
#pragma unroll
        for (int i = 0; i < RKEY_WORDS; ++i) same &= *reinterpret_cast<volatile uint64_t *>(&B->key[i]) == key[i];
        if (same) {
            if ((c >> 8) != tag) return R_DEAD;
            if (*reinterpret_cast<volatile unsigned int *>(&B->tinv) > tinv) return R_DEAD;
            atomicMax(&B->tinv, tinv);
            return (uint32_t)b;
        }
        if (++b == nb) b = 0;
    }
    atomicExch(error, 1u);
    return R_DEAD;
}
__global__ void __launch_bounds__(TILE) rb_rehash_kernel(const RBucket *__restrict__ old_table, uint64_t old_nb,
                                                         RBucket *__restrict__ table, uint64_t nb, Counters *ctr) {
    const uint64_t i = (uint64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= old_nb || old_table[i].ctrl == 0) return;
    uint64_t key[RKEY_WORDS];
#pragma unroll
    for (int k = 0; k < RKEY_WORDS; ++k) key[k] = old_table[i].key[k];
    const uint32_t game = old_table[i].pad;
    uint64_t b = __umul64hi(rb_key_hash(key, game), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        if (atomicCAS(&table[b].ctrl, 0ull, old_table[i].ctrl) == 0) {
#pragma unroll
            for (int k = 0; k < RKEY_WORDS; ++k) table[b].key[k] = key[k];
            table[b].pad = game;
            return;
        }
        if (++b == nb) b = 0;
    }
    atomicExch(&ctr->error, 1u);
}

// goal test on dequeue (:827-829), per game: goal[g] = first rank inside game g whose game is over
__global__ void __launch_bounds__(TILE) rb_goal_kernel(const RRec *__restrict__ front, int64_t n, const int64_t *__restrict__ seg,
                                                       int n_games, const RConfigDev *__restrict__ cfg, long long *__restrict__ goal) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    const int g = rb_game_of(seg, n_games, i);
    const RPlayer p = front[i].p[front[i].cur];
    if (r_pts(cfg[g], p) >= cfg[g].target) atomicMin(goal + g, (long long)(i - seg[g]));
}

// r_count_scan_kernel over the batch queue; the parents of a game whose goal was found this level get no successors.
// cands[g] += successors of game g.
__global__ void __launch_bounds__(TILE) rb_count_scan_kernel(const RRec *__restrict__ front, int64_t n, const int64_t *__restrict__ seg,
                                                             int n_games, const RConfigDev *__restrict__ cfg,
                                                             const long long *__restrict__ goal, uint32_t *__restrict__ off,
                                                             uint32_t *__restrict__ vmask, uint64_t *status, Counters *ctr, int ticket_id,
                                                             unsigned long long *cands) {
    __shared__ uint32_t warp_sums[TILE / 32 + 1];
    __shared__ uint32_t s_tile;
    __shared__ uint64_t s_base;
    if (threadIdx.x == 0) s_tile = atomicAdd(&ctr->ticket[ticket_id], 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const int64_t p = (int64_t)tile * TILE + threadIdx.x;
    uint32_t cnt = 0, m = 0;
    int g = -1;
    if (p < n) {
        g = rb_game_of(seg, n_games, p);
        if (goal[g] == 0x7fffffffffffffffll) {
            RRec s;
            ld_rec(front + p, s);
            int bonus[NCOL], pts;
            r_derive(cfg[g], s.p[s.cur], bonus, pts);
            m = r_valid_mask(cfg[g], s, bonus);
            cnt = __popc(m);
        }
        vmask[p] = m;
    }
    rb_warp_add(cands, g, cnt);
    uint32_t total;
    const uint32_t excl = block_excl_scan(cnt, warp_sums, total);
    if (threadIdx.x < 32) {
        const uint64_t e = lookback_exclusive(status, tile, total, 0);
        if (threadIdx.x == 0) {
            s_base = e;
            if ((int64_t)(tile + 1) * TILE >= n) ctr->total_cands = e + total;
        }
    }
    __syncthreads();
    if (p < n) off[p] = (uint32_t)(s_base + excl);
}

// r_expand_kernel over the batch queue: link = rank of the parent inside its game << 8 | ordinal; cand_game[t] = game
__global__ void __launch_bounds__(TILE) rb_expand_kernel(const RRec *__restrict__ front, int64_t n, const int64_t *__restrict__ seg,
                                                         int n_games, const RConfigDev *__restrict__ cfg,
                                                         const uint32_t *__restrict__ off, const uint32_t *__restrict__ vmask,
                                                         RRec *__restrict__ cand, uint32_t *__restrict__ cand_game) {
    const int64_t p = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (p >= n) return;
    uint32_t m = vmask[p], ord = 0;
    if (!m) return;
    const int g = rb_game_of(seg, n_games, p);
    RRec s;
    ld_rec(front + p, s);
    int bonus[NCOL], pts;
    r_derive(cfg[g], s.p[s.cur], bonus, pts);
    uint64_t t = off[p];
    const uint64_t rank = (uint64_t)(p - seg[g]);
    while (m) {
        const int slot = __ffs(m) - 1;
        m &= m - 1;
        RRec o;
        r_make_child(cfg[g], s, bonus, slot, o);
        o.link = (rank << 8) | ord;
        o.spare = 0;
        st_rec(cand + t, o);
        cand_game[t] = (uint32_t)g;
        ++t;
        ++ord;
    }
}

// exact-key probe / insert of the batch's candidates, (game, key) identity; n_new[g] += new states of game g
__global__ void __launch_bounds__(TILE) rb_probe_kernel(const RRec *__restrict__ cand, const uint32_t *__restrict__ cand_game, int64_t n,
                                                        const RConfigDev *__restrict__ cfg, RBucket *__restrict__ table, uint64_t nb,
                                                        uint64_t tag, uint32_t *__restrict__ cand_slot, Counters *ctr,
                                                        unsigned long long *n_new_game) {
    const int64_t t = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint32_t n_new = 0;
    int g = -1;
    if (t < n) {
        g = (int)cand_game[t];
        RRec s;
        ld_rec(cand + t, s);
        uint64_t key[RKEY_WORDS];
        if (!r_pack_key(cfg[g], s, key)) atomicExch(&ctr->error, 4u);
        cand_slot[t] = rb_probe(table, nb, tag, key, (uint32_t)g, ~(uint32_t)t, n_new, &ctr->error);
    }
    rb_warp_add(n_new_game, g, n_new);
#pragma unroll
    for (int d = 16; d; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
    if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(&ctr->n_new, (unsigned long long)n_new);
}

// the winners' records and games, in arrival order
__global__ void __launch_bounds__(TILE) rb_gather_kernel(const RRec *__restrict__ src, const uint32_t *__restrict__ src_game,
                                                         const int64_t *__restrict__ idx, int64_t n, RRec *__restrict__ dst,
                                                         uint32_t *__restrict__ dst_game) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        const int64_t j = idx[i];
        RRec r;
        ld_rec(src + j, r);
        st_rec(dst + i, r);
        dst_game[i] = src_game[j];
    }
}

// sort pairs of the beam cut: y[i] = ~flip_f64(score) (ascending y = descending score), slot[i] = i; score key range
// in ctr->sk_min / sk_max
__global__ void __launch_bounds__(TILE) rb_score_kernel(const RRec *__restrict__ recs, const uint32_t *__restrict__ games, int64_t n,
                                                        const RConfigDev *__restrict__ cfg, ScoreLuts L, uint64_t *__restrict__ y,
                                                        uint32_t *__restrict__ slot, Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint64_t kmin = ~0ull, kmax = 0;
    if (i < n) {
        RRec s;
        ld_rec(recs + i, s);
        const uint64_t k = flip_f64((uint64_t)__double_as_longlong(r_score(cfg[games[i]], s, L)));
        y[i] = ~k;
        slot[i] = (uint32_t)i;
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
// sort word of the second (game) pass: the game of each pair, in the score order the first pass left
__global__ void __launch_bounds__(TILE) rb_game_words_kernel(const uint32_t *__restrict__ slot, const uint32_t *__restrict__ games,
                                                             int64_t n, uint64_t *__restrict__ y) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) y[i] = games[slot[i]];
}
// segmented cut: the pairs are in (game, score desc, arrival) order; pair i is rank i - useg[g] of game g and is kept
// at kseg[g] + rank when that rank is below kseg[g + 1] - kseg[g] = min(beam_g, unique_g)
__global__ void __launch_bounds__(TILE) rb_cut_kernel(const RRec *__restrict__ uniq, const uint32_t *__restrict__ games,
                                                      const uint32_t *__restrict__ slot, int64_t n, const int64_t *__restrict__ useg,
                                                      const int64_t *__restrict__ kseg, RRec *__restrict__ front) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = slot[i];
    const int g = (int)games[j];
    const int64_t r = i - useg[g];
    if (r < kseg[g + 1] - kseg[g]) {
        RRec rec;
        ld_rec(uniq + j, rec);
        st_rec(front + kseg[g] + r, rec);
    }
}

// out[i] = col[at[i]]: the link words of the games' path states at one level
__global__ void __launch_bounds__(TILE) rb_pick_kernel(const uint64_t *__restrict__ col, const int64_t *__restrict__ at, int64_t n,
                                                       uint64_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) out[i] = col[at[i]];
}

// every game's line, one thread per game: out[g][0] = root, out[g][p + 1] = successor ords[g][p] of out[g][p]
// (the reference's list(iter(state))[ordinal]) for p < plies[g]
__global__ void __launch_bounds__(TILE) rb_line_kernel(const RRec *__restrict__ roots, const RConfigDev *__restrict__ cfg, int n_games,
                                                       const int32_t *__restrict__ plies, const uint8_t *__restrict__ ords,
                                                       int max_plies, RRec *__restrict__ out, Counters *ctr) {
    const int g = blockIdx.x * TILE + threadIdx.x;
    if (g >= n_games) return;
    const RConfigDev &C = cfg[g];
    RRec s;
    ld_rec(roots + g, s);
    RRec *line = out + (int64_t)g * (max_plies + 1);
    st_rec(line, s);
    for (int p = 0; p < plies[g]; ++p) {
        int bonus[NCOL], pts;
        r_derive(C, s.p[s.cur], bonus, pts);
        uint32_t m = r_valid_mask(C, s, bonus);
        const int ord = ords[(int64_t)g * max_plies + p];
        if (ord >= __popc(m)) {
            atomicExch(&ctr->error, 1u);
            return;
        }
        for (int k = 0; k < ord; ++k) m &= m - 1;
        RRec o;
        r_make_child(C, s, bonus, __ffs(m) - 1, o);
        o.link = (uint64_t)ord;
        o.spare = 0;
        st_rec(line + p + 1, o);
        s = o;
    }
}

}  // namespace spl
