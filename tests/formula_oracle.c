/* formula_oracle.c -- CPU oracle of formula heuristics (splendor-rl-gym_b200/formula.py).  TEST INFRASTRUCTURE ONLY.
 *
 * Built by tests/formula_oracle.py into a temporary directory.  It compiles the oracle (oracle/splendor_oracle.c, used
 * as it is) into the same library and adds what formulas need on top of it:
 *   orcf_score        t_i = ((coef * x1 ** e1) * x2 ** e2) * x3 ** e3, score = ((t_0 + t_1) + ...) + randint * 0.01,
 *                     C pow and separately rounded * and + (-ffp-contract=off), as CPython evaluates the expression
 *   orcf_solver_step  one level of the oracle's solver scored by a formula: the oracle's own step as exhaustive BFS
 *                     (expansion, first-arrival dedup, goal test, links), then the beam cut of src/solver.py:452-456
 *                     -- sorted(next_queue, key=formula, reverse=True)[:beam] -- with the oracle's stable merge sort. */
#include "../oracle/splendor_oracle.c"

typedef struct {
    double coef;
    int32_t n_factors;
    int32_t feature[3]; /* 0 pts, 1 saved, 2 cards, 3 sum(gems), 4 sum(bonus), 5 sum(gems) + 2 sum(bonus), 6 bonus colours,
                           7 + c gems[c], 12 + c bonus[c] */
    double exponent[3];
} orcf_term;
typedef struct {
    int32_t n_terms, reserved;
    orcf_term term[8];
} orcf_formula;

static int orcf_feature(const orc_state *s, int f) {
    int sum_g = 0, sum_b = 0, nnz = 0;
    unsigned gk = st_gems(s);
    for (int c = 0; c < NCOL; c++) {
        sum_g += (gk >> (3 * c)) & 7;
        sum_b += st_bonus(s, c);
        nnz += st_bonus(s, c) > 0;
    }
    switch (f) {
    case 0: return st_pts(s);
    case 1: return st_saved(s);
    case 2: return st_ncards(s);
    case 3: return sum_g;
    case 4: return sum_b;
    case 5: return sum_g + 2 * sum_b;
    case 6: return nnz;
    default: return f < 12 ? (int)((gk >> (3 * (f - 7))) & 7) : st_bonus(s, f - 12);
    }
}

/* noise_mode 0 const, 1 hash; r_ext > 0: that randint value instead */
double orcf_score(const orc_state *s, const orcf_formula *F, int noise_mode, int r_ext) {
    volatile double acc = 0.0, t;
    for (int i = 0; i < F->n_terms; i++) {
        const orcf_term *T = &F->term[i];
        t = T->coef;
        for (int j = 0; j < T->n_factors; j++) t = t * pow((double)orcf_feature(s, T->feature[j]), T->exponent[j]);
        acc = i ? acc + t : t;
    }
    double noise = r_ext > 0 ? (double)r_ext * 0.01 : noise_of(s, noise_mode);
    acc = acc + noise;
    return acc;
}

/* S was created with use_heuristic = 1; its built-in heuristic id is not used */
int orcf_solver_step(orc_solver *S, const orcf_formula *F, orc_level_info *info) {
    S->use_heuristic = 0;
    int done = orc_solver_step(S, info);
    S->use_heuristic = 1;
    if (done) return 1;
    orc_level *L = &S->levels[S->nlevels - 1];
    int64_t n = L->n;
    double *sc = (double *)malloc(n * 8);
    int64_t *idx = (int64_t *)malloc(n * 8), *tmp = (int64_t *)malloc(n * 8);
    for (int64_t i = 0; i < n; i++) { sc[i] = orcf_score(&L->st[i], F, S->noise_mode, 0); idx[i] = i; }
    g_score = sc; g_st = L->st; g_policy = S->policy;
    msort(idx, tmp, n);
    int64_t k = n < S->beam ? n : S->beam;
    orc_state *kx = (orc_state *)malloc(k * sizeof(orc_state));
    uint64_t *kl = (uint64_t *)malloc(k * 8);
    for (int64_t i = 0; i < k; i++) { kx[i] = L->st[idx[i]]; kl[i] = L->link[idx[i]]; }
    free(L->st); free(L->link); free(sc); free(idx); free(tmp);
    L->st = kx; L->link = kl; L->n = k;
    if (info) info->kept = k;
    return 0;
}
