/*
 * splendor_b200.h -- C ABI of the B200-native frontier-expansion library
 * (libsplendor_b200.so, built from splendor-rl-gym_b200/csrc/ for sm_100a).
 *
 * This is the drop-in boundary for ONE path of IamJasonBian/Splendor-RL-Gym: the
 * per-turn frontier expansion of its solver (generate -> dedup -> score -> top-k).
 * Every entry point names the reference interface (file:line in the reference tree)
 * it replaces.  Plain pointers and sizes only: no torch / C++ types cross this line.
 *
 * Conventions
 *   - every function returns an int32 status: 0 = ok, < 0 = SPL_E_* ; the message of
 *     the last failure on a context is spl_last_error(ctx) (spl_last_error(NULL) for
 *     failures of spl_create itself).  No C++ exception crosses the boundary.
 *   - "dev" pointers are CUDA device pointers owned by the caller (e.g. torch tensors);
 *     "host" pointers are ordinary host memory.  `stream` is a cudaStream_t passed as
 *     void* (NULL = the legacy default stream).  Calls are asynchronous on `stream`
 *     unless they return a count through a host pointer, in which case they
 *     synchronise that stream before returning.
 *   - one context per device, used from one host thread at a time.
 *   - there is NO CPU fallback: on a machine without a usable sm_100 device every
 *     compute entry point fails with SPL_E_NODEVICE / SPL_E_CUDA.
 *
 * Packed state record (speedrun `State`, src/solver.py:308-318)
 *   key  (spl_key, 128 bit, identity == (cards, gems) exactly as hashed at :318):
 *        bits 0..14   gems[c] << 3c          (c = White, Blue, Green, Red, Black; 0..7 each)
 *        bits 15..104 card i owned -> bit 15+i   (90 cards, src/cardparser.py:57-66)
 *        bits 105..127 zero in caller-visible keys (used as epoch tag inside the visited table)
 *        Unsigned 128-bit order of keys == order of the Python int
 *        (sum(1 << card) << 15) | sum(gems[i] << 3i)  used by the `det` tie-break policy.
 *   aux  (uint64, NOT part of identity -- first arrival supplies it, src/solver.py:447-450):
 *        bits 0..15 saved | bits 16..23 pts | bits 24+5c..28+5c bonus[c]
 *   link (uint64): parent_rank << 8 | ordinal, ordinal = index into list(iter(parent))
 *        (buys of affordable not-owned cards in ascending card index, then takes in
 *        table order; src/solver.py:357-388).
 */
#ifndef SPLENDOR_B200_H
#define SPLENDOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPL_ABI_VERSION 2

typedef struct spl_ctx spl_ctx;
typedef struct spl_solver spl_solver;

typedef struct { uint64_t lo, hi; } spl_key;

/* status codes */
enum {
    SPL_OK = 0,
    SPL_E_INVALID = -1,    /* bad argument */
    SPL_E_NODEVICE = -2,   /* no CUDA device / not an sm_100 device */
    SPL_E_CUDA = -3,       /* CUDA runtime error (message has the detail) */
    SPL_E_NOMEM = -4,      /* device allocation failed */
    SPL_E_TABLE_FULL = -5, /* visited table cannot take this level (grow failed) */
    SPL_E_CAPACITY = -6,   /* caller buffer too small */
    SPL_E_STATE = -7       /* call out of order (e.g. step after the search ended) */
};

/* heuristic ids == the reference registry HEURISTICS (src/solver.py:299-305);
 * unknown names map to SIMPLE on the host side, as HEURISTICS.get(name, simple) does (:429). */
enum { SPL_H_SIMPLE = 0, SPL_H_BALANCED = 1, SPL_H_AGGRESSIVE = 2, SPL_H_EFFICIENCY = 3 };

/* noise policy for the `randint(1,100)*0.01` term (src/solver.py:215,247,260,284), SURVEY.md 8a-N */
enum {
    SPL_NOISE_CONST = 0,    /* randint -> 50 */
    SPL_NOISE_HASH = 1,     /* randint -> 1 + splitmix64(lo^hi) % 100 */
    SPL_NOISE_EXTERNAL = 2  /* the i-th state scored in a level (arrival order) gets the i-th randint(1, 100) of a
                             * host-side stream, e.g. the reference's own seeded Mersenne Twister: see spl_solver_cut */
};

/* tie-break policy of the beam cut `sorted(next_queue, key=h, reverse=True)[:beam]` (:452-456) */
enum { SPL_TIE_STABLE = 0 /* arrival order, as Python's stable sort */, SPL_TIE_KEY = 1 /* key descending */,
       /* spl_dtopk_cut only: threshold by key as SPL_TIE_KEY, and the caller guarantees that the local keys are already in
        * descending order by index (the sharded driver's arrival keys), so the local rank sort orders by score alone */
       SPL_TIE_KEY_ORDERED = 2 };
/* what makes two speedrun states "the same" for the visited set (spl_set_identity) */
enum { SPL_IDENT_KEY = 0 /* exact 105-bit (cards, gems) key */, SPL_IDENT_PYHASH = 1 /* the reference's hash((cards, gems)) */ };

typedef struct {
    int32_t device;            /* CUDA device ordinal */
    int32_t reserved0;
    uint64_t table_slots;      /* initial visited-table capacity in slots: three per 64-byte bucket, at most
                                * 3 * 2^30 (0 = default 2^22) */
    uint64_t max_table_bytes;  /* growth ceiling for the visited table (0 = 60% of free device memory) */
    uint64_t chunk_parents;    /* parents expanded per round (0 = default: 4 Mi on the key-table level, 16 Mi on the
                                * card-set-grouped level; max 16 Mi) */
    uint64_t node_slots;       /* initial capacity of the card-set node table (384-byte nodes) used by the beam-search
                                * level (0 = default 2^12; grows by rehash) */
    uint64_t max_node_bytes;   /* growth ceiling of the node table (0 = 50% of free device memory) */
} spl_config;

/* per-level counters (the reference prints none of these; they feed parity tests and the roofline) */
typedef struct {
    int32_t level;        /* index of the `while queue` iteration (src/solver.py:434) */
    int32_t ended;        /* 1 when the loop ended in this iteration (goal dequeued / frontier empty) */
    int64_t frontier;     /* len(queue) at the top of the iteration */
    int64_t expanded;     /* parents actually expanded on the device */
    int64_t generated;    /* successors enumerated (== sum of len(list(parent))) */
    int64_t unique;       /* len(next_queue): first arrivals not in the visited set */
    int64_t kept;         /* len(queue) after the beam cut */
    int64_t goal_rank;    /* rank of the first state with pts >= goal in queue order, or -1 */
    int64_t visited;      /* len(trail) */
    uint64_t table_slots; /* current visited-table capacity */
    /* CUDA-event times of the level's stages.  Key-table level (BFS, pyhash, mt noise) | card-set-grouped level (beam): */
    float ms_count;       /* fan-out count + offset scan                 | fan-out count + buy records */
    float ms_expand;      /* expand+probe launches (dominant kernel)     | per-run dedup: thread + warp + CTA kernels */
    float ms_resolve;     /* resolve+emit(+score) launches               | item sort + run boundaries (grouping) */
    float ms_select;      /* ... of the radix-select + cut */
    float ms_sort;        /* ... of the rank-ordering sort + gather */
    float ms_warp;        /* grouped level: the warp kernel alone (the dominant kernel of ms_expand) */
} spl_level_info;

/* ---- library / context ------------------------------------------------------------------ */
int32_t spl_abi_version(void);
const char *spl_last_error(const spl_ctx *ctx);

/* Host-only table access (no device needed).  The tables are built once, natively, from
 * the packed deck; they replace get_deck() (src/cardparser.py:64), get_takes()
 * (src/gems.py:111-113) and possible_buys()/get_buys() (src/buys.py:13-17,39-41). */
const uint32_t *spl_deck_table(int32_t *n_cards);                     /* cost|pt|bonus per card */
int32_t spl_host_takes(const uint8_t gems[5], uint8_t out[100 * 5]);  /* -> count, take_gems order */
int32_t spl_host_buys(const uint8_t key[5], uint8_t out[90]);         /* -> count, ascending cards */

int32_t spl_create(const spl_config *cfg, spl_ctx **out);
int32_t spl_destroy(spl_ctx *ctx);
/* forget every visited state (trail = {}), keep the allocation */
int32_t spl_reset_visited(spl_ctx *ctx, void *stream);

/* Identity of the speedrun solver's visited set (`trail`, src/solver.py:426, :447-449).  SPL_IDENT_KEY
 * (default): the exact (cards, gems) key.  SPL_IDENT_PYHASH: the reference's own State.hash =
 * hash((cards, gems)) (src/solver.py:316; State.__eq__ compares only that value, :335-336) -- two states
 * whose 64-bit CPython hashes collide are merged, first arrival wins, exactly as the reference's dict does.
 * Applies to solvers created afterwards on this context (speedrun solver only; stage operators and
 * realistic mode keep their own identities).  SURVEY.md 8(f).3. */
int32_t spl_set_identity(spl_ctx *ctx, int32_t identity);

/* Parent links of the kept states (`trail[state] = parent`, src/solver.py:449; walked back from the goal at
 * :459-464) are held as one 8-byte column per level.  Solvers created afterwards on this context keep at most
 * `device_bytes` of them in HBM (0 = no limit, the default): past that the oldest levels move to pinned host memory
 * and spl_solver_path / spl_gs_link_at read them there.  SURVEY.md 8(f).2.  spl_spilled_bytes: bytes moved so far
 * (they are also counted by spl_transfer_bytes). */
int32_t spl_set_link_budget(spl_ctx *ctx, uint64_t device_bytes);
int32_t spl_spilled_bytes(spl_ctx *ctx, int64_t *n_host);

/* out[i] = hash((cards, gems)) of keys[i] as CPython computes it (unsigned 64-bit view); device buffers.
 * Replaces: State.__init__'s `self.hash = hash((self.cards, self.gems))`, src/solver.py:316. */
int32_t spl_pyhash(spl_ctx *ctx, const spl_key *keys_dev, int64_t n, uint64_t *out_dev, void *stream);
int32_t spl_visited_count(spl_ctx *ctx, int64_t *n_host);
/* kernels launched by this context so far (bench.py's gpu_launches) */
int32_t spl_launch_count(spl_ctx *ctx, int64_t *n_host);
/* host<->device bytes copied by this context so far (bench.py's e2e accounting) */
int32_t spl_transfer_bytes(spl_ctx *ctx, int64_t *h2d_host, int64_t *d2h_host);

/* Device buffers that the other processes of this node can map (CUDA IPC), for spl_gs_round_buys_peer: the owner
 * allocates and publishes the 64-byte handle, every peer opens it once (peer access over NVLink is enabled on open). */
int32_t spl_ipc_alloc(spl_ctx *ctx, uint64_t bytes, void **ptr_dev_out, uint8_t handle_out[64]);
int32_t spl_ipc_open(spl_ctx *ctx, const uint8_t handle[64], void **ptr_dev_out);
int32_t spl_ipc_close(spl_ctx *ctx, void *ptr_dev);
int32_t spl_ipc_free(spl_ctx *ctx, void *ptr_dev);

/* ---- stage operators (caller-owned device buffers) ---------------------------------------- */

/* State.__iter__ for a batch (src/solver.py:357-388): all successors of parents
 * [0, n) in (parent rank, ordinal) order.  cand_link[j] = parent_rank << 8 | ordinal.
 * Fails with SPL_E_CAPACITY (and reports the needed size in *n_out_host) if cap is too small. */
int32_t spl_expand(spl_ctx *ctx, const spl_key *keys_dev, const uint64_t *aux_dev, int64_t n,
                   spl_key *cand_keys_dev, uint64_t *cand_aux_dev, uint64_t *cand_link_dev,
                   int64_t cap, int64_t *n_out_host, void *stream);

/* `if next_step in trail: continue; trail[next_step] = puzzle; next_queue.append(next_step)`
 * (src/solver.py:447-450) for a candidate list given in arrival order: keeps the FIRST
 * arrival of every key never seen before (in this call or any earlier one on this
 * context), in arrival order.  uniq_src[j] = index of the surviving candidate. */
int32_t spl_dedup(spl_ctx *ctx, const spl_key *cand_keys_dev, const uint64_t *cand_aux_dev, int64_t n,
                  spl_key *uniq_keys_dev, uint64_t *uniq_aux_dev, int64_t *uniq_src_dev,
                  int64_t *n_out_host, void *stream);

/* HEURISTICS[name](state) for a batch (src/solver.py:210-286), bit-exact IEEE doubles. */
int32_t spl_score(spl_ctx *ctx, int32_t heuristic, int32_t noise, const spl_key *keys_dev,
                  const uint64_t *aux_dev, int64_t n, double *scores_dev, void *stream);

/* sorted(range(n), key=score, reverse=True)[:k] (src/solver.py:452-456) under a tie policy:
 * writes the surviving indices in rank order. */
int32_t spl_topk(spl_ctx *ctx, const double *scores_dev, const spl_key *keys_dev, int64_t n, int64_t k,
                 int32_t tie_policy, int64_t *out_idx_dev, int64_t *n_out_host, void *stream);

/* ---- multi-GPU building blocks (one process per GPU; the collectives themselves are issued by the
 * host through torch.distributed/NCCL between these calls) -------------------------------------
 * The reference has no distributed path; these exist so that a frontier sharded by key hash
 * across ranks produces bit-identical levels to the single-GPU solver (SURVEY.md 8e). */

/* stable partition of a candidate list by owner rank = f(key) mod n_ranks: perm_dev[j] = index of the
 * j-th candidate in (owner, arrival) order; counts_host[g] = candidates owned by rank g. */
int32_t spl_owner_partition(spl_ctx *ctx, const spl_key *keys_dev, int64_t n, int32_t n_ranks, int64_t *perm_dev,
                            int64_t *counts_host, void *stream);

/* Row-based variants for the sharded driver (rows = 32-byte records {lo, hi, aux, link}):
 *   spl_expand_rows     successors of front rows, link = (rank_base + parent) << 8 | ordinal
 *   spl_route_keys      send buffer = candidate keys in (owner, arrival) order + per-owner counts;
 *                       the permutation stays in the context for spl_compact_winners
 *   spl_dedup_flags     owner side: first-arrival dedup of a received key list -> one winner byte each
 *   spl_compact_winners source side: winner bytes (in send order) -> the winning rows in arrival order */
int32_t spl_expand_rows(spl_ctx *ctx, const void *front_rows_dev, int64_t n, int64_t rank_base, void *out_rows_dev,
                        int64_t cap, int64_t *n_out_host, void *stream);
int32_t spl_route_keys(spl_ctx *ctx, const void *cand_rows_dev, int64_t n, int32_t n_ranks, spl_key *send_keys_dev,
                       int64_t *counts_host, void *stream);
int32_t spl_dedup_flags(spl_ctx *ctx, const spl_key *keys_dev, int64_t n, uint8_t *flags_dev, void *stream);
int32_t spl_compact_winners(spl_ctx *ctx, const void *cand_rows_dev, int64_t n, const uint8_t *flags_send_order_dev,
                            void *out_rows_dev, int64_t *n_out_host, void *stream);

/* HEURISTICS[name] over rows; out[i] = rows[idx[i]] (scatter = 0) or out[idx[i]] = rows[i] (scatter = 1) */
int32_t spl_score_rows(spl_ctx *ctx, int32_t heuristic, int32_t noise, const void *rows_dev, int64_t n, double *scores_dev,
                       const uint8_t *draws_dev_or_null /* SPL_NOISE_EXTERNAL: randint value per row */, void *stream);
int32_t spl_move_rows(spl_ctx *ctx, const void *rows_dev, const int64_t *idx_dev, int64_t n, void *out_rows_dev,
                      int32_t scatter, void *stream);

/* distributed beam cut: the radix select of spl_topk, one pass at a time, so that the host can
 * all-reduce the 2048-bin histogram (*hist_dev_out, uint32) between spl_dtopk_hist and spl_dtopk_pick.
 * word 0 = score passes, word 1/2 = key.hi / key.lo passes among score ties (det policy).  The key array
 * given to spl_dtopk_begin is read in place by the later passes: keep it alive until spl_dtopk_cut. */
int32_t spl_dtopk_begin(spl_ctx *ctx, const double *scores_dev, const spl_key *keys_dev_or_null, int64_t n,
                        uint64_t *sk_min_host, uint64_t *sk_max_host, void *stream);
int32_t spl_dtopk_hist(spl_ctx *ctx, int32_t word, int32_t shift, int32_t bits, int32_t first, uint64_t sk_min_global,
                       uint32_t **hist_dev_out, void *stream);
int32_t spl_dtopk_pick(spl_ctx *ctx, int32_t word, int32_t shift, int32_t first, int32_t init_k, int64_t k, void *stream);
/* select state = {score threshold (x space), tie quota, count above, tie bucket size, key.hi, key.lo threshold} */
int32_t spl_dtopk_get(spl_ctx *ctx, uint64_t state_host[6], void *stream);
int32_t spl_dtopk_set(spl_ctx *ctx, const uint64_t state_host[6], void *stream);
/* local cut by the state set above + local rank sort; outputs the survivors' indices and sort words */
int32_t spl_dtopk_cut(spl_ctx *ctx, int32_t tie_policy, int32_t keep_all, int32_t all_ties, uint64_t sk_min_global,
                      uint64_t sk_max_global, int64_t *out_idx_dev, uint64_t *out_y_dev, uint64_t *out_klo_dev,
                      uint64_t *out_khi_dev, int64_t *kept_host, void *stream);
/* out[i] (+)= #{ j : b[j] < a[i] } (or <= when inclusive) for ascending-sorted composite b; words = 1 | 3;
 * sorted_a = 1 promises that a is ascending too (lets each CTA bracket its slice of a inside b first) */
int32_t spl_count_less(spl_ctx *ctx, int32_t words, int32_t inclusive, const uint64_t *ay_dev, const uint64_t *akl_dev,
                       const uint64_t *akh_dev, int64_t na, const uint64_t *by_dev, const uint64_t *bkl_dev,
                       const uint64_t *bkh_dev, int64_t nb, int64_t *out_dev, int32_t accumulate, int32_t sorted_a,
                       void *stream);

/* ---- fused level-synchronous solver: State.solve (src/solver.py:390-464) ------------------- */

/* root_host: one packed state (key + aux) in HOST memory -- the `self` of solve().
 * use_heuristic = 0 -> exhaustive BFS (queue = next_queue); else beam search. */
int32_t spl_solver_create(spl_ctx *ctx, const spl_key *root_key_host, uint64_t root_aux_host,
                          int32_t goal_pts, int32_t use_heuristic, int32_t heuristic, int64_t beam_width,
                          int32_t tie_policy, int32_t noise, int32_t keep_links, spl_solver **out);
/* The same solve from a level-0 queue of n_rows >= 1 packed rows {lo, hi, aux, link} (32 bytes each, HOST memory) in
 * rank order; the link words are ignored.  Every row is registered as visited (trail = {row: None for row in rows}),
 * and spl_solver_path ends at the rank of the row the goal descends from.  spl_solver_create is this call with its
 * root as the only row.  SPL_E_INVALID, naming the row, for an illegal gem hand (a colour above 7 or more than 10
 * gems), a key bit at or above 105, or two rows with the same key. */
int32_t spl_solver_create_queue(spl_ctx *ctx, const void *rows_host, int64_t n_rows, int32_t goal_pts,
                                int32_t use_heuristic, int32_t heuristic, int64_t beam_width, int32_t tie_policy,
                                int32_t noise, int32_t keep_links, spl_solver **out);
int32_t spl_solver_destroy(spl_solver *s);
/* one `while queue` iteration; returns SPL_OK and fills *info_host; info->ended tells the caller to stop */
int32_t spl_solver_step(spl_solver *s, spl_level_info *info_host, void *stream);
/* SPL_NOISE_EXTERNAL only: spl_solver_step stops after expand + dedup with info->kept == -1 and
 * info->unique == the number of states to score; the host then supplies that many draws (uint8, each the
 * value randint(1, 100) returned, in arrival order) and this call scores, cuts and sorts the level. */
int32_t spl_solver_cut(spl_solver *s, const uint8_t *draws_dev, int64_t n_draws, spl_level_info *info_host, void *stream);
/* device views of the current queue (valid until the next step) */
int32_t spl_solver_frontier(spl_solver *s, const spl_key **keys_dev, const uint64_t **aux_dev,
                            const uint64_t **link_dev, int64_t *n_host);
/* parent-chain walk (src/solver.py:459-464): ordinals[i] = index into list(iter(path[i])) of
 * path[i+1]; ranks[i] = rank of path[i] in level i.  Returns the number of moves in *n_moves_host. */
int32_t spl_solver_path(spl_solver *s, int64_t *ranks_host, int32_t *ordinals_host, int32_t cap,
                        int32_t *n_moves_host);

/* ---- sharded beam search: queue sharded BY CARD SET, one process per GPU (csrc/spl_shard.cuh) -------------------
 * The reference has no distributed path (SURVEY.md 5, 8e); these entry points spread State.solve's level loop
 * (src/solver.py:434-457) over `world` ranks so that every level holds the same states, in the same order, as on one
 * GPU.  A queue state lives on the rank that owns its cards; its gem-take successors (same cards, :381-388) are
 * deduplicated on that GPU, card buys (:369-374) are written as 32-byte records {key, aux, link} into per-destination
 * ranges of a send buffer.  The collectives themselves (all-to-all of the records, all-gather of the score
 * dictionaries, all-reduce of the tie histograms, sample sort of the survivors' sort words) are issued by the host
 * between these calls (torch.distributed / NCCL).  Policy: ties by arrival order, noise const | hash. */
typedef struct spl_gsolver spl_gsolver;
int32_t spl_gs_create(spl_ctx *ctx, int32_t rank, int32_t world, const spl_key *root_key_host, uint64_t root_aux_host,
                      int32_t goal_pts, int32_t heuristic, int64_t beam_width, int32_t noise, int32_t keep_links,
                      spl_gsolver **out);
int32_t spl_gs_destroy(spl_gsolver *s);
/* goal test on dequeue (:443-445): GLOBAL rank of the first local queue state with pts >= goal (INT64_MAX: none) */
int32_t spl_gs_goal(spl_gsolver *s, int64_t *rank_host, int64_t *n_local_host, void *stream);
/* round = the local parents with global rank in [rank_lo, rank_hi): fan-out and the number of buy records this rank
 * sends to every rank (counts_host[world]) */
int32_t spl_gs_round_begin(spl_gsolver *s, int64_t rank_lo, int64_t rank_hi, int64_t *counts_host, int64_t *n_parents_host,
                           void *stream);
/* the round's buy records into send_dev (destination d owns [sum(counts[0..d)), +counts[d])) */
int32_t spl_gs_round_buys(spl_gsolver *s, void *send_dev, void *stream);
/* the same records stored straight into the receive buffers of their owners over NVLink peer mappings (the store is
 * the transfer; no send buffer, no all-to-all): recv_dev_of_rank[d] = rank d's receive buffer as mapped into this
 * process (spl_ipc_open; this rank's own buffer for d == rank), offset_at_rank[d] = records of lower ranks that
 * precede this rank's there (sum of counts[r][d], r < rank).  Callers fence with a stream-ordered collective before
 * anyone reads its buffer. */
int32_t spl_gs_round_buys_peer(spl_gsolver *s, void *const *recv_dev_of_rank, const int64_t *offset_at_rank, void *stream);
/* owner side (:447-450): local parents + the n_recv records received -> first-arrival dedup per card set, winners + scores */
int32_t spl_gs_round_group(spl_gsolver *s, const void *recv_dev, int64_t n_recv, int64_t *n_new_host, void *stream);
int32_t spl_gs_counters(spl_gsolver *s, int64_t *n_uniq_host, int64_t *generated_host, int64_t *visited_host);
/* CUDA-event times of the level's owner-side stages: item sort + runs, thread kernel, warp kernel, CTA kernel */
int32_t spl_gs_stage_ms(spl_gsolver *s, float ms_host[4]);
/* beam cut (:452-456) across ranks: local score dictionary -> (host all-gathers) -> global threshold ... */
int32_t spl_gs_dict(spl_gsolver *s, void **dict_dev, int64_t *bytes_host, void *stream);
int32_t spl_gs_threshold(spl_gsolver *s, const void *dicts_dev, int64_t k, int64_t n_uniq_global, int32_t *need_ties_host,
                         void *stream);
/* ... ties of the threshold score split by arrival order: radix select over the ranks' tie words; the host
 * all-reduces *hist_dev (2048 x uint32) between spl_gs_tie_hist and spl_gs_tie_pick ... */
int32_t spl_gs_tie_begin(spl_gsolver *s, int32_t *link_bits_host, void *stream);
int32_t spl_gs_tie_hist(spl_gsolver *s, int32_t shift, int32_t bits, int32_t first, uint32_t **hist_dev, void *stream);
int32_t spl_gs_tie_pick(spl_gsolver *s, int32_t shift, int32_t first, void *stream);
/* ... local cut + local sort by the sort word (score rank << link bits | link; a total order over all ranks) */
int32_t spl_gs_cut(spl_gsolver *s, int32_t have_tie_threshold, int64_t *kept_local_host, const uint64_t **y_sorted_dev,
                   int32_t *y_bits_host, void *stream);
/* global ranks of the survivors (= queue order of the next level): sample sort of the sort words */
int32_t spl_gs_partition(spl_gsolver *s, const uint64_t *probes_host, int32_t n_probes, int64_t *bounds_host, void *stream);
int32_t spl_gs_rank_sort(spl_gsolver *s, const uint64_t *y_dev, int64_t n, int32_t y_bits, int64_t base, int64_t *ranks_out_dev,
                         void *stream);
int32_t spl_gs_adopt(spl_gsolver *s, const int64_t *granks_dev, int64_t n_global_next, void *stream);
int32_t spl_gs_frontier(spl_gsolver *s, const void **recs_dev, const uint64_t **granks_dev, int64_t *n_local_host);
/* parent chain (:459-464): link of the state with global rank `grank` in the queue of `level`, if this rank holds it */
int32_t spl_gs_link_at(spl_gsolver *s, int32_t level, int64_t grank, int32_t *found_host, uint64_t *link_host);

/* ---- realistic multi-player mode: MultiPlayerState (src/solver.py:471-860) ---------------------
 * State record = 96 bytes:
 *   struct { uint64 mlo; uint32 mhi; uint16 gems; uint16 saved; } p[4];   card mask / gems (3 b per colour) / saved
 *   uint8 vis[12];  visible card per market slot in slot order, tier-major (255 = empty)
 *   uint8 cur; uint8 pad[3]; uint64 link; uint64 spare;
 * bonus, pts, gem pool, deck position and final-round state are derived (see csrc/spl_realistic.cuh).
 * The visited set of this mode is keyed by the EXACT identity (spl_rpack: 384-bit packing), 64-byte buckets.
 * The market order is an INPUT: deck[t] = full sequence of tier t (visible cards first), as built by
 * CardMarket.from_full_deck(shuffle, seed) (src/solver.py:94-119) on the host. */
typedef struct {
    int32_t num_players;     /* 2..4  (GameConfig.num_players, src/solver.py:29) */
    int32_t target_points;   /* GameConfig.target_points */
    int32_t gems_per_color;  /* GameConfig.gems_per_color: 4 / 5 / 7 */
    int32_t noise;           /* SPL_NOISE_* for the randint term at :810 */
    int32_t deck_len[3];
    uint8_t deck[3][40];
} spl_rconfig;

/* MultiPlayerState.__iter__ (:568-748) for a batch of records: successors in reference order
 * (buys in market slot order, colour triples in combinations() order, double takes). */
int32_t spl_rexpand(spl_ctx *ctx, const spl_rconfig *cfg, const void *recs_dev, int64_t n, void *out_recs_dev,
                    int64_t cap, int64_t *n_out_host, void *stream);
/* multi_competitive_heuristic (:778-812), bit-exact doubles */
int32_t spl_rscore(spl_ctx *ctx, const spl_rconfig *cfg, const void *recs_dev, int64_t n, double *scores_dev, void *stream);
/* The exact identity key of realistic mode (src/solver.py:495-500, PlayerState :177-186): 6 x uint64 per record --
 * card owner codes, gems and saved per player, deck position of every visible slot, current player (injective; the
 * reference's own identity is a 64-bit hash of the same fields).  keys_out_dev[n][6]. */
int32_t spl_rpack(spl_ctx *ctx, const spl_rconfig *cfg, const void *recs_dev, int64_t n, uint64_t *keys_out_dev, void *stream);
/* max(p.pts for p in state.players) per record: the progress line at :832-836 */
int32_t spl_rmaxpts(spl_ctx *ctx, const spl_rconfig *cfg, const void *recs_dev, int64_t n, uint8_t *out_dev, void *stream);
/* MultiPlayerState.solve (:750-860): beam always applied, ties by arrival order, game over when play
 * returns to the player who triggered the final round.  Steps / path / destroy via spl_solver_*.  This is the
 * single-GPU search; a search spread over several GPUs runs only when asked (see the key-sharded block below). */
int32_t spl_rsolver_create(spl_ctx *ctx, const spl_rconfig *cfg, const void *root_rec_host, int64_t beam_width,
                           int32_t keep_links, spl_solver **out);
int32_t spl_rsolver_frontier(spl_solver *s, const void **recs_dev, int64_t *n_host);

/* ---- batched realistic search (realistic.py: solve_many) -------------------------------------------------------------
 * n_games independent MultiPlayerState.solve() searches advance in lockstep on one GPU: each spl_solver_step is one level
 * of every game still running, at a number of kernel launches that does not depend on n_games.  Game g has its own
 * rules, market (cfgs[g]), root record (root_recs_host[g], 96 bytes) and beam width (beams[g] >= 1); noise must be
 * SPL_NOISE_CONST or SPL_NOISE_HASH (SPL_E_INVALID otherwise: the draws of 'mt' depend on the other games).  Every level
 * of game g equals spl_rsolver's level for that game alone: the same records in the same rank order (link words carry
 * ranks inside the game), the same counters, goal rank and line.  A state of one game never merges with a state of
 * another: the visited identity is (game, exact key).  A game leaves the batch when its goal is dequeued, its queue
 * runs out or it reaches the 1000-turn limit; the batch ends when every game has.  spl_solver_step fills the aggregate
 * counters over the games of the level (frontier, generated, unique, kept: sums; visited: the batch's table; goal_rank
 * -1; ended when every game has) with ms_count = goal test + count, ms_expand = expand, ms_resolve = probe + winners,
 * ms_select = score, ms_sort = the segmented cut.  A level above 2^32 - 1 candidates fails with SPL_E_INVALID; a full
 * visited table or device memory fails with SPL_E_TABLE_FULL / SPL_E_NOMEM, and the context stays usable once the
 * solver is destroyed.  Destroy with spl_solver_destroy; spl_solver_path does not apply (use spl_rbatch_lines). */
typedef struct {
    int64_t level;      /* the last level the game took part in */
    int64_t frontier;   /* its queue length at the top of that level */
    int64_t generated, unique, kept, visited;  /* as spl_level_info, for this game alone */
    int64_t goal_rank;  /* rank of its first finished state in that queue, or -1 */
    int32_t ended;      /* 1 once the game has ended (its counters no longer change) */
    int32_t pad;
} spl_rgame_info;
int32_t spl_rbatch_create(spl_ctx *ctx, const spl_rconfig *cfgs, const void *root_recs_host, const int64_t *beams,
                          int32_t n_games, int32_t keep_links, spl_solver **out);
/* the per-game counters after the last spl_solver_step (n_games must be the batch's) */
int32_t spl_rbatch_games(spl_solver *s, spl_rgame_info *out_host, int32_t n_games);
/* game `game`'s queue (its records in rank order, device memory of the solver); empty once the game has ended */
int32_t spl_rbatch_frontier(spl_solver *s, int32_t game, const void **recs_dev, int64_t *n_host);
/* after the batch has ended (keep_links = 1): every game's line, root first.  plies_host[g] = moves of game g; its
 * plies_host[g] + 1 records go to recs_host[g * cap ...].  SPL_E_CAPACITY (plies_host filled) when a line needs more
 * than cap records.  The lines are rebuilt on the device from the link columns, one thread per game. */
int32_t spl_rbatch_lines(spl_solver *s, void *recs_host, int64_t cap, int32_t *plies_host);

/* ---- batched speedrun search (solver.py: State.solve_many) --------------------------------------------------------
 * n_games independent State.solve() searches advance in lockstep on one GPU: each spl_solver_step is one level of every
 * game still running, at a number of kernel launches that does not depend on n_games.  Game g starts from the 32-byte
 * row root_rows_host[g] = {lo, hi, aux, link} (link ignored) and has its own goal (goals[g]), search kind
 * (use_heuristic[g]: 0 = exhaustive BFS, every unique state in arrival order) and, for beam search, heuristic
 * (heuristics[g], as spl_solver_create's) and beam width (beams[g] >= 1).  tie_policy (SPL_TIE_STABLE or SPL_TIE_KEY)
 * and noise (SPL_NOISE_CONST or SPL_NOISE_HASH: externally drawn noise would depend on the other games) hold for the
 * whole batch.  Every root is checked as spl_solver_create_queue checks its rows (illegal gem hand, key bit at or
 * above 105); equal roots in different games are separate games.  A bad root, beam, tie policy or noise fails with
 * SPL_E_INVALID, naming the game.  Every level of game g equals spl_solver_create's level for that game alone: the
 * same rows in the same rank order (link words carry ranks inside the game), the same counters, goal rank and line.
 * A state of one game never merges with a state of another: the visited identity is (game, key).  A game leaves the
 * batch when a state of its queue meets its goal or its queue runs out (there is no turn limit, as in State.solve);
 * the batch ends when every game has.  spl_solver_step fills the aggregate counters as for spl_rbatch_create, with
 * ms_select = score and ms_sort = the key passes ('det') and the segmented cut.  A level above 2^32 - 1 candidates
 * fails with SPL_E_INVALID; a full visited table or device memory fails with SPL_E_TABLE_FULL / SPL_E_NOMEM, and the
 * context stays usable once the solver is destroyed.  Destroy with spl_solver_destroy; spl_solver_path does not apply
 * (use spl_sbatch_lines).  Link columns spill past spl_set_link_budget as a single solve's do. */
int32_t spl_sbatch_create(spl_ctx *ctx, const void *root_rows_host /* n_games x {lo, hi, aux, link} */, const int32_t *goals,
                          const int32_t *use_heuristic, const int32_t *heuristics, const int64_t *beams, int32_t n_games,
                          int32_t tie_policy, int32_t noise, int32_t keep_links, spl_solver **out);
/* the per-game counters after the last spl_solver_step (n_games must be the batch's) */
int32_t spl_sbatch_games(spl_solver *s, spl_rgame_info *out_host, int32_t n_games);
/* game `game`'s queue as 32-byte rows {lo, hi, aux, link} in rank order (device memory of the solver; link = parent
 * rank inside the game << 8 | ordinal); empty once the game has ended */
int32_t spl_sbatch_frontier(spl_solver *s, int32_t game, const void **rows_dev, int64_t *n_host);
/* after the batch has ended (keep_links = 1): every game's line, root first, as 32-byte rows (link = the ordinal that
 * leads to the row, ~0 for the root).  plies_host[g] = moves of game g; its plies_host[g] + 1 rows go to
 * rows_host[g * cap ...].  SPL_E_CAPACITY (plies_host filled) when a line needs more than cap rows. */
int32_t spl_sbatch_lines(spl_solver *s, void *rows_host, int64_t cap, int32_t *plies_host);

/* ---- realistic mode on the key-sharded driver (sharded.py: RCudaBackend + RShardedSolver) ---------------------------
 * MultiPlayerState.solve(shard=True) / --realistic --shard: the level loop of :820-852 over a queue spread block-cyclically
 * across ranks, with the same per-level steps as spl_expand_rows .. spl_move_rows above.  Every level holds the same
 * records, in the same order, as spl_rsolver.  Ties by arrival order, noise const | hash (the config's; spl_rscore scores
 * the records).  Realistic mode shards only when asked.  Each spl_r* row call is its speedrun twin on 96-byte records and
 * 384-bit identity keys, with these differences:
 *   spl_rexpand_rows     successors follow :568-748 under the config; rank_base must be >= 0
 *   spl_rroute_keys      send_keys_dev[n][6] holds the packed keys (spl_rpack); owner = low 32 bits of the key hash, the
 *                        owner's bucket comes from the high bits.  SPL_E_INVALID when a key cannot be packed.  Its
 *                        permutation is kept apart from spl_route_keys': only spl_rcompact_winners may follow it
 *   spl_rdedup_flags     (:840-843) inserts into the realistic visited table, which grows as spl_rsolver's does;
 *                        SPL_E_TABLE_FULL when it cannot take the list (no state is dropped)
 *   spl_rcompact_winners SPL_E_STATE unless it follows spl_rroute_keys on the same candidates
 *   spl_rmove_rows       96-byte records
 *   spl_rfirst_goal      first queue index whose game is over (:827-829: players[cur].pts >= target), -1 if none
 *   spl_rreset_visited   forget every visited state of the context: the realistic table and, as spl_rsolver_create does,
 *                        the speedrun table (spl_reset_visited clears only that one).  The epoch counter restarts, so a
 *                        long-lived context never runs out of epochs; each spl_rdedup_flags call takes one (at most
 *                        2^23 - 1 calls between two resets)
 *   spl_rvisited_count   states in the realistic visited table (spl_visited_count counts the speedrun table's) */
int32_t spl_rexpand_rows(spl_ctx *ctx, const spl_rconfig *cfg, const void *front_recs_dev, int64_t n, int64_t rank_base,
                         void *out_recs_dev, int64_t cap, int64_t *n_out_host, void *stream);
int32_t spl_rroute_keys(spl_ctx *ctx, const spl_rconfig *cfg, const void *cand_recs_dev, int64_t n, int32_t n_ranks,
                        uint64_t *send_keys_dev, int64_t *counts_host, void *stream);
int32_t spl_rdedup_flags(spl_ctx *ctx, const uint64_t *keys_dev, int64_t n, uint8_t *flags_dev, void *stream);
int32_t spl_rcompact_winners(spl_ctx *ctx, const void *cand_recs_dev, int64_t n, const uint8_t *flags_send_order_dev,
                             void *out_recs_dev, int64_t *n_out_host, void *stream);
int32_t spl_rmove_rows(spl_ctx *ctx, const void *recs_dev, const int64_t *idx_dev, int64_t n, void *out_recs_dev,
                       int32_t scatter, void *stream);
int32_t spl_rfirst_goal(spl_ctx *ctx, const spl_rconfig *cfg, const void *front_recs_dev, int64_t n, int64_t *rank_host,
                        void *stream);
int32_t spl_rreset_visited(spl_ctx *ctx, void *stream);
int32_t spl_rvisited_count(spl_ctx *ctx, int64_t *n_host);

#ifdef __cplusplus
}
#endif
#endif /* SPLENDOR_B200_H */
