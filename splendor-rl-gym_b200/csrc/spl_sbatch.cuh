// spl_sbatch.cuh -- the sm_100a kernels of the batched speedrun search (spl_sbatch_*): B State.solve() searches in
// lockstep on one GPU.
//
// The layout is the batched realistic search's (spl_realistic.cuh, rb_*): every per-record array of a level is
// game-major, game g owning the index range seg[g] .. seg[g + 1], and inside it the records keep the order the
// single-game solver gives them.  Link words carry the parent's rank inside its game, so each game's segment of the
// queue is byte-identical to the queue of spl_solver_create for that game alone.  gm[g] is game g's goal, search kind
// and heuristic.  Successors, payments and scores come from the speedrun device functions of spl_kernels.cuh
// (derive_parent, make_child, score_state): the rules are not restated here.
#pragma once
#include "spl_kernels.cuh"
#include "spl_realistic.cuh"

namespace spl {

struct SGame {
    int32_t goal;       // points that end the game when a state with them is dequeued
    int32_t use_h;      // 0: exhaustive BFS (every unique state, arrival order), 1: beam search
    int32_t heuristic;  // score_state's h
    int32_t pad;
};

// Visited table of the batch: 32-byte buckets, one state each: {key.lo, key.hi | game << 41, ctrl, ~t, pad}.  The
// key-table slot of spl_kernels.cuh has no room for the game (its bits 105..127 are the epoch tag), so this table keeps
// the game beside the 105-bit key and compares both.  ctrl and ~t work as in RBucket: ctrl = tag << 8 | 1 while the
// claimer writes the key, tag << 8 | 3 once it is readable; atomicMax of ~t keeps the first arrival.  The game is mixed
// into the bucket hash: the games of a heuristic or beam sweep from one root share every early state, and without the
// mixing each such state would be one probe run B buckets deep.
struct __align__(32) SBucket {
    uint64_t lo, hi_game;
    unsigned long long ctrl;
    unsigned int tinv, pad;
};
static_assert(sizeof(SBucket) == 32, "SBucket layout");
constexpr int SB_GAME_SHIFT = 41;  // hi_game = key bits 64..104 | game << 41

__device__ __forceinline__ uint64_t sb_key_hash(uint64_t lo, uint64_t hi_game) {
    return mix64(hash_key(lo, hi_game & HI_KEY_MASK), 0x9E3779B97F4A7C15ull * ((hi_game >> SB_GAME_SHIFT) + 1));
}

__device__ __forceinline__ uint32_t sb_probe(SBucket *__restrict__ table, uint64_t nb, uint64_t tag, uint64_t lo, uint64_t hi_game,
                                             uint32_t tinv, uint32_t &n_new, unsigned int *error) {
    uint64_t b = __umul64hi(sb_key_hash(lo, hi_game), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        SBucket *B = table + b;
        unsigned long long c = *reinterpret_cast<volatile unsigned long long *>(&B->ctrl);
        if (c == 0) {
            c = atomicCAS(&B->ctrl, 0ull, (unsigned long long)(tag << 8 | 1));
            if (c == 0) {  // claimed: write the key, then publish
                B->lo = lo;
                B->hi_game = hi_game;
                __threadfence();
                atomicExch(&B->ctrl, (unsigned long long)(tag << 8 | 3));
                ++n_new;
                atomicMax(&B->tinv, tinv);
                return (uint32_t)b;
            }
        }
        while ((c & 3) == 1) c = *reinterpret_cast<volatile unsigned long long *>(&B->ctrl);  // key not published yet
        __threadfence();
        if (*reinterpret_cast<volatile uint64_t *>(&B->lo) == lo && *reinterpret_cast<volatile uint64_t *>(&B->hi_game) == hi_game) {
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

// move every ready bucket of an old table into a larger one (tags preserved)
__global__ void __launch_bounds__(TILE) sb_rehash_kernel(const SBucket *__restrict__ old_table, uint64_t old_nb,
                                                         SBucket *__restrict__ table, uint64_t nb, Counters *ctr) {
    const uint64_t i = (uint64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= old_nb || old_table[i].ctrl == 0) return;
    const uint64_t lo = old_table[i].lo, hg = old_table[i].hi_game;
    uint64_t b = __umul64hi(sb_key_hash(lo, hg), nb);
    for (int probes = 0; probes < MAX_PROBE; ++probes) {
        if (atomicCAS(&table[b].ctrl, 0ull, old_table[i].ctrl) == 0) {
            table[b].lo = lo;
            table[b].hi_game = hg;
            return;
        }
        if (++b == nb) b = 0;
    }
    atomicExch(&ctr->error, 1u);
}

// goal test on the queue (src/solver.py:443-445), per game: goal[g] = first rank inside game g with pts >= its goal
__global__ void __launch_bounds__(TILE) sb_goal_kernel(const Rec *__restrict__ front, int64_t n, const int64_t *__restrict__ seg,
                                                       int n_games, const SGame *__restrict__ gm, long long *__restrict__ goal) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    const int g = rb_game_of(seg, n_games, i);
    if ((int)((front[i].aux >> 16) & 0xff) >= gm[g].goal) atomicMin(goal + g, (long long)(i - seg[g]));
}

// count_scan_kernel over the batch queue; the parents of a game whose goal was found this level get no successors.
// cands[g] += successors of game g.
__global__ void __launch_bounds__(TILE) sb_count_scan_kernel(const Rec *__restrict__ front, int64_t n, const int64_t *__restrict__ seg,
                                                             int n_games, const long long *__restrict__ goal,
                                                             const DevTables *__restrict__ tabs, const uint32_t *__restrict__ takes_idx,
                                                             uint32_t *__restrict__ off, uint64_t *status, Counters *ctr, int ticket_id,
                                                             unsigned long long *cands) {
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
    int g = -1;
    if (p < n) {
        g = rb_game_of(seg, n_games, p);
        if (goal[g] == 0x7fffffffffffffffll) {
            Rec r;
            ld_rec(front + p, r);
            uint64_t bl, bh;
            uint32_t nb, tk;
            derive_parent(s, takes_idx, r.lo, r.hi, r.aux, bl, bh, nb, tk);
            cnt = nb + (tk & 0xff);
        }
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

// successors of the batch queue in list(iter(parent)) order, one parent per thread: cand[off[p] + ord] with link =
// rank of the parent inside its game << 8 | ord, and its game in cand_game
__global__ void __launch_bounds__(TILE) sb_expand_kernel(const Rec *__restrict__ front, int64_t n, const int64_t *__restrict__ seg,
                                                         int n_games, const long long *__restrict__ goal,
                                                         const DevTables *__restrict__ tabs, const uint32_t *__restrict__ takes_idx,
                                                         const uint16_t *__restrict__ takes_edges, const uint32_t *__restrict__ off,
                                                         Rec *__restrict__ cand, uint32_t *__restrict__ cand_game) {
    __shared__ SmemTabs s;
    load_tabs(s, tabs);
    __syncthreads();
    const int64_t p = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (p >= n) return;
    const int g = rb_game_of(seg, n_games, p);
    if (goal[g] != 0x7fffffffffffffffll) return;
    Rec r;
    ld_rec(front + p, r);
    uint64_t bl, bh;
    uint32_t nb, tk;
    derive_parent(s, takes_idx, r.lo, r.hi, r.aux, bl, bh, nb, tk);
    const uint32_t cnt = nb + (tk & 0xff);
    const uint64_t t = off[p], rank = (uint64_t)(p - seg[g]);
    for (uint32_t ord = 0; ord < cnt; ++ord) {
        Rec o;
        make_child(s, takes_edges, r.lo, r.hi, r.aux, bl, bh, nb, tk, ord, o.lo, o.hi, o.aux);
        o.link = rank << 8 | ord;
        st_rec(cand + t + ord, o);
        cand_game[t + ord] = (uint32_t)g;
    }
}

// (game, key) probe / insert of the batch's candidates (arrival index = list index); n_new[g] += new states of game g
__global__ void __launch_bounds__(TILE) sb_probe_kernel(const Rec *__restrict__ cand, const uint32_t *__restrict__ cand_game, int64_t n,
                                                        SBucket *__restrict__ table, uint64_t nb, uint64_t tag,
                                                        uint32_t *__restrict__ cand_slot, Counters *ctr, unsigned long long *n_new_game) {
    const int64_t t = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint32_t n_new = 0;
    int g = -1;
    if (t < n) {
        g = (int)cand_game[t];
        uint64_t lo, hi;
        ld_cg_u64x2(reinterpret_cast<const uint64_t *>(cand + t), lo, hi);
        cand_slot[t] = sb_probe(table, nb, tag, lo, (hi & HI_KEY_MASK) | (uint64_t)g << SB_GAME_SHIFT, ~(uint32_t)t, n_new, &ctr->error);
    }
    rb_warp_add(n_new_game, g, n_new);
#pragma unroll
    for (int d = 16; d; d >>= 1) n_new += __shfl_xor_sync(0xffffffffu, n_new, d);
    if ((threadIdx.x & 31) == 0 && n_new) atomicAdd(&ctr->n_new, (unsigned long long)n_new);
}

// winners (first arrivals of new states) in arrival order: out_idx[rank] = list index; 8 candidates per thread.
// r_winners_kernel's ticketed scan over the batch table's buckets.
__global__ void __launch_bounds__(TILE) sb_winners_kernel(const uint32_t *__restrict__ cand_slot, const SBucket *__restrict__ table,
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

// the winners' records and games, in arrival order
__global__ void __launch_bounds__(TILE) sb_gather_kernel(const Rec *__restrict__ src, const uint32_t *__restrict__ src_game,
                                                         const int64_t *__restrict__ idx, int64_t n, Rec *__restrict__ dst,
                                                         uint32_t *__restrict__ dst_game) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        const int64_t j = idx[i];
        Rec r;
        ld_rec(src + j, r);
        st_rec(dst + i, r);
        dst_game[i] = src_game[j];
    }
}

// sort pairs of the beam cut: y[i] = ~flip_f64(score) (ascending y = descending score; score_kernel's f64 for the
// game's heuristic and `noise`), or 0 for a game of exhaustive BFS, whose arrival order the stable passes then keep;
// slot[i] = i.  ctr->sk_min / sk_max: the range of flip_f64(score); ctr->key_or / key_and: which key bits vary (the
// 'det' policy's key passes).  Both over the beam games only.
__global__ void __launch_bounds__(TILE) sb_score_kernel(const Rec *__restrict__ recs, const uint32_t *__restrict__ games, int64_t n,
                                                        const SGame *__restrict__ gm, int noise_mode, ScoreLuts L,
                                                        uint64_t *__restrict__ y, uint32_t *__restrict__ slot, Counters *ctr) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    uint64_t kmin = ~0ull, kmax = 0, or_lo = 0, or_hi = 0, and_lo = ~0ull, and_hi = ~0ull;
    if (i < n) {
        Rec r;
        ld_rec(recs + i, r);
        const SGame G = gm[games[i]];
        uint64_t w = 0;
        if (G.use_h) {
            const uint64_t k = flip_f64((uint64_t)__double_as_longlong(score_state(G.heuristic, noise_mode, r.lo, r.hi & HI_KEY_MASK, r.aux, L)));
            w = ~k;
            kmin = kmax = k;
            or_lo = and_lo = r.lo;
            or_hi = and_hi = r.hi & HI_KEY_MASK;
        }
        y[i] = w;
        slot[i] = (uint32_t)i;
    }
#pragma unroll
    for (int d = 16; d; d >>= 1) {
        kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, d));
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, d));
        or_lo |= __shfl_xor_sync(0xffffffffu, or_lo, d);
        or_hi |= __shfl_xor_sync(0xffffffffu, or_hi, d);
        and_lo &= __shfl_xor_sync(0xffffffffu, and_lo, d);
        and_hi &= __shfl_xor_sync(0xffffffffu, and_hi, d);
    }
    if ((threadIdx.x & 31) == 0 && kmin <= kmax) {
        atomicMin(&ctr->sk_min, (unsigned long long)kmin);
        atomicMax(&ctr->sk_max, (unsigned long long)kmax);
        atomicOr(&ctr->key_or[0], (unsigned long long)or_lo);
        atomicOr(&ctr->key_or[1], (unsigned long long)or_hi);
        atomicAnd(&ctr->key_and[0], (unsigned long long)and_lo);
        atomicAnd(&ctr->key_and[1], (unsigned long long)and_hi);
    }
}

// sort word of one pass, in the order the earlier passes left: y[i] = src[slot[i] * stride] ^ flip for a beam game's
// pair, 0 for a BFS game's (the 'det' policy's key words ~key.lo / ~key.hi, then the score words saved aside)
__global__ void __launch_bounds__(TILE) sb_words_kernel(const uint32_t *__restrict__ slot, int64_t n, const uint64_t *__restrict__ src,
                                                        int stride, uint64_t flip, const uint32_t *__restrict__ games,
                                                        const SGame *__restrict__ gm, uint64_t *__restrict__ y) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i < n) {
        const uint32_t j = slot[i];
        y[i] = gm[games[j]].use_h ? src[(int64_t)j * stride] ^ flip : 0;
    }
}

// segmented cut (rb_cut_kernel for 32-byte rows): the pairs are in (game, rank) order; pair i is rank i - useg[g] of
// game g and is kept at kseg[g] + rank when that rank is below kseg[g + 1] - kseg[g] = min(beam_g, unique_g)
__global__ void __launch_bounds__(TILE) sb_cut_kernel(const Rec *__restrict__ uniq, const uint32_t *__restrict__ games,
                                                      const uint32_t *__restrict__ slot, int64_t n, const int64_t *__restrict__ useg,
                                                      const int64_t *__restrict__ kseg, Rec *__restrict__ front) {
    const int64_t i = (int64_t)blockIdx.x * TILE + threadIdx.x;
    if (i >= n) return;
    const uint32_t j = slot[i];
    const int g = (int)games[j];
    const int64_t r = i - useg[g];
    if (r < kseg[g + 1] - kseg[g]) {
        Rec rec;
        ld_rec(uniq + j, rec);
        st_rec(front + kseg[g] + r, rec);
    }
}

// every game's line, one thread per game: out[g][0] = root, out[g][p + 1] = successor ords[g][p] of out[g][p]
// (the reference's list(iter(state))[ordinal]) for p < plies[g]; link = the ordinal
__global__ void __launch_bounds__(TILE) sb_line_kernel(const Rec *__restrict__ roots, int n_games, const int32_t *__restrict__ plies,
                                                       const uint8_t *__restrict__ ords, int max_plies, const DevTables *__restrict__ tabs,
                                                       const uint32_t *__restrict__ takes_idx, const uint16_t *__restrict__ takes_edges,
                                                       Rec *__restrict__ out, Counters *ctr) {
    __shared__ SmemTabs s;
    load_tabs(s, tabs);
    __syncthreads();
    const int g = blockIdx.x * TILE + threadIdx.x;
    if (g >= n_games) return;
    Rec r;
    ld_rec(roots + g, r);
    Rec *line = out + (int64_t)g * (max_plies + 1);
    st_rec(line, r);
    for (int p = 0; p < plies[g]; ++p) {
        uint64_t bl, bh;
        uint32_t nb, tk;
        derive_parent(s, takes_idx, r.lo, r.hi, r.aux, bl, bh, nb, tk);
        const uint32_t ord = ords[(int64_t)g * max_plies + p];
        if (ord >= nb + (tk & 0xff)) {
            atomicExch(&ctr->error, 1u);
            return;
        }
        Rec o;
        make_child(s, takes_edges, r.lo, r.hi, r.aux, bl, bh, nb, tk, ord, o.lo, o.hi, o.aux);
        o.link = ord;
        st_rec(line + p + 1, o);
        r = o;
    }
}

}  // namespace spl
