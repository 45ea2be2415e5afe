// spl_common.cuh -- shared types and device helpers of the sm_100a frontier-expansion library.
//
// Data layout in HBM (see DESIGN.md):
//   frontier record  : 32 B AoS {lo, hi, aux, link}  -> one 256-bit load per parent
//   visited-table bucket: 64 B = one DRAM burst = three slots: sector 0 {lo0, hi0|tag, ~t0 ~t1 ~t2 (u32), spare},
//                         sector 1 {lo1, hi1|tag, lo2, hi2|tag}
//   candidate slot id : u32 per generated successor, in (parent rank, ordinal) order
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "deck_table.h"

namespace spl {

constexpr int NCOL = 5;
constexpr int TILE = 256;               // parents per CTA tile == threads per CTA
constexpr uint32_t DEAD = 0xFFFFFFFFu;  // candidate already in the visited set (earlier epoch)
constexpr uint64_t GEM_MASK = 0x7FFFull;
constexpr int GEM_STATES = 2898;     // gem hands with every colour <= 7 and at most 10 gems
constexpr int NODE_BM_WORDS = 46;    // 2944 bits >= GEM_STATES: one bit per gem hand, in gemrank order
constexpr uint64_t HI_KEY_MASK = (1ull << 41) - 1;  // key bits 64..104
constexpr int TAG_SHIFT = 41;                       // epoch tag in bits 105..127 of the table slot
constexpr uint32_t TAG_MAX = (1u << 23) - 1;
constexpr int MAX_PROBE = 1 << 14;

struct __align__(32) Rec {  // frontier record
    uint64_t lo, hi, aux, link;
};

// Constant tables built on the host (spl_tables.cuh) and uploaded once per context.
struct DevTables {
    // possible-buys table in separable form (src/buys.py:13-17): a card is affordable iff for
    // every colour c its cost[c] <= min(gems[c] + bonus[c], 7), so buys[k] = AND_c M[c][k_c].
    // Masks are stored in KEY bit layout (card i at key bit 15+i) -> {lo, hi}.
    uint64_t buy_lo[NCOL][8];
    uint64_t buy_hi[NCOL][8];
    uint32_t card[SPL_NUM_CARDS];  // packed cost|pt|bonus (deck_table.h)
};

// A registered formula heuristic (spl_add_formula) as the device reads it; the context's formulas sit in one table,
// id SPL_H_FORMULA_BASE + k at index k, which the kernels that can score formulas take as their last parameter (so the
// parameters of the built-in kernels keep their layout).  Every factor points at the power table of its (feature,
// exponent) pair, pw[x] = pow(x, exponent) over the feature's whole domain.
struct FormFactor {
    const double *pw;
    int32_t feat;  // SPL_F_*
    int32_t pad;
};
struct FormTerm {
    double coef;
    int32_t nf, pad;
    FormFactor f[SPL_FORMULA_MAX_FACTORS];
};
struct FormDev {
    int32_t nt, pad[3];
    FormTerm t[SPL_FORMULA_MAX_TERMS];
};

struct ScoreLuts {  // x ** e for every integer argument the heuristics can see (src/solver.py:210-286)
    const double *pts;    // [4][256]   pts ** {2.5, 2.8, 3.2, 2.0}
    const double *saved;  // [4][65536] saved ** {0.4, 0.5, 0.3, 0.7}
    const double *small;  // [6][512]: 0: res**0.3, 1: ncards**0.6, 2: nnz**0.4, 3: sumb**0.5, 4: sumb**1.2, 5: nnz**0.8
};

// ------------------------------------------------------------------ memory helpers
__device__ __forceinline__ void ld_cg_u64x2(const uint64_t *p, uint64_t &a, uint64_t &b) {
    asm volatile("ld.global.cg.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p));
}
// one 32-byte sector of a visited-table bucket in one request (LDG.E.256.STRONG.GPU)
__device__ __forceinline__ void ld_u64x4_cg(const uint64_t *p, uint64_t &a, uint64_t &b, uint64_t &c, uint64_t &d) {
    asm volatile("ld.global.cg.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
}
// the {lo, hi|tag} words of slot j of bucket B (16-byte aligned: the operand of the 128-bit CAS)
template <typename T>
__device__ __forceinline__ T *bucket_key(T *B, int j) { return B + (j ? 2 + 2 * j : 0); }
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t *p) {
    uint32_t a;
    asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(a) : "l"(p));
    return a;
}
constexpr int BUCKET_SLOTS = 3;
// candidate verdict / slot id = bucket << 2 | slot-in-bucket (buckets < 2^30); the slot's ~t word
__device__ __forceinline__ const uint32_t *slot_tword(const uint64_t *table, uint32_t sid) {
    return reinterpret_cast<const uint32_t *>(table + ((uint64_t)(sid >> 2) << 3) + 2) + (sid & 3);
}
__device__ __forceinline__ void ld_rec(const Rec *p, Rec &r) {  // 256-bit load (LDG.E.256 on sm_100)
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0, %1, %2, %3}, [%4];"
                 : "=l"(r.lo), "=l"(r.hi), "=l"(r.aux), "=l"(r.link)
                 : "l"(p));
}
// four consecutive u64 of a read-only stream (32-byte aligned)
__device__ __forceinline__ void ld_u64x4(const uint64_t *p, uint64_t &a, uint64_t &b, uint64_t &c, uint64_t &d) {
    asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(a), "=l"(b), "=l"(c), "=l"(d) : "l"(p));
}
__device__ __forceinline__ void st_rec(Rec *p, const Rec &r) {
    asm volatile("st.global.v4.u64 [%0], {%1, %2, %3, %4};" ::"l"(p), "l"(r.lo), "l"(r.hi), "l"(r.aux), "l"(r.link)
                 : "memory");
}
// 128-bit compare-and-swap on a visited-table slot (ATOMG.E.CAS.128 on sm_90+)
__device__ __forceinline__ void cas128(uint64_t *addr, uint64_t clo, uint64_t chi, uint64_t slo, uint64_t shi,
                                       uint64_t &olo, uint64_t &ohi) {
    asm volatile(
        "{\n .reg .b128 c, s, d;\n mov.b128 c, {%2, %3};\n mov.b128 s, {%4, %5};\n"
        " atom.relaxed.gpu.global.cas.b128 d, [%6], c, s;\n mov.b128 {%0, %1}, d;\n}\n"
        : "=l"(olo), "=l"(ohi)
        : "l"(clo), "l"(chi), "l"(slo), "l"(shi), "l"(addr)
        : "memory");
}

// ------------------------------------------------------------------ hashing
__device__ __host__ __forceinline__ uint64_t hash_key(uint64_t lo, uint64_t hi) {
    uint64_t x = lo ^ (hi * 0x9E3779B97F4A7C15ull);
    x ^= x >> 32;
    x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32;
    x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32;
    return x;
}
// home bucket of a key among `nb` buckets
__device__ __forceinline__ uint64_t slot_of(uint64_t h, uint64_t nb) { return __umul64hi(h, nb); }

// splitmix64 finaliser over the folded key: noise policy `hash` (SURVEY.md 8a-N)
__device__ __host__ __forceinline__ uint64_t mix64(uint64_t lo, uint64_t hi) {
    uint64_t x = lo ^ hi;
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// order-preserving map double -> u64 (larger double <=> larger u64; handles negative scores)
// -0.0 is canonicalised to +0.0 first: Python's sort compares them equal (ties -> arrival order).
__device__ __host__ __forceinline__ uint64_t flip_f64(uint64_t b) {
    if (b == 0x8000000000000000ull) b = 0;
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __host__ __forceinline__ uint64_t unflip_f64(uint64_t k) { return (k >> 63) ? (k & 0x7FFFFFFFFFFFFFFFull) : ~k; }

// ------------------------------------------------------------------ block primitives (TILE threads)
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v) {
    const unsigned lane = threadIdx.x & 31;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        uint32_t t = __shfl_up_sync(0xffffffffu, v, d);
        if (lane >= d) v += t;
    }
    return v;
}
// exclusive scan of one u32 per thread over the CTA; returns the exclusive prefix, total in `total`
__device__ __forceinline__ uint32_t block_excl_scan(uint32_t v, uint32_t *warp_sums /*[TILE/32 + 1]*/, uint32_t &total) {
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t inc = warp_incl_scan(v);
    if (lane == 31) warp_sums[w] = inc;
    __syncthreads();
    if (w == 0) {
        uint32_t s = lane < TILE / 32 ? warp_sums[lane] : 0;
        uint32_t si = warp_incl_scan(s);
        if (lane < TILE / 32) warp_sums[lane] = si - s;
        if (lane == TILE / 32 - 1) warp_sums[TILE / 32] = si;
    }
    __syncthreads();
    uint32_t r = inc - v + warp_sums[w];
    total = warp_sums[TILE / 32];
    __syncthreads();
    return r;
}

// Decoupled look-back over tiles that were handed out by an atomic ticket (so every
// predecessor tile is already resident).  status word = flag << 62 | value;
// flag 1 = tile aggregate published, 2 = inclusive prefix published.  Called by ALL 32 lanes of
// warp 0 (converged); every lane gets the result.  The warp inspects 32 predecessors per step, so a
// deep window of aggregate-only tiles costs one L2 round trip per 32 tiles instead of one per tile.
__device__ __forceinline__ uint64_t lookback_exclusive(volatile uint64_t *status, uint32_t tile, uint64_t aggregate,
                                                       uint64_t base0) {
    constexpr uint64_t VAL = (1ull << 62) - 1;
    const unsigned lane = threadIdx.x & 31;
    if (tile == 0) {
        if (lane == 0) status[0] = (2ull << 62) | ((base0 + aggregate) & VAL);
        return base0;
    }
    if (lane == 0) status[tile] = (1ull << 62) | (aggregate & VAL);
    uint64_t excl = 0;
    for (int64_t j = (int64_t)tile - 1;; j -= 32) {
        const int64_t idx = j - lane;  // lane 0 = nearest predecessor; idx < 0 = before tile 0 (which always ends the walk)
        uint64_t s;
        do { s = idx >= 0 ? status[idx] : (2ull << 62); } while (__any_sync(0xffffffffu, (s >> 62) == 0));
        const unsigned incl = __ballot_sync(0xffffffffu, (s >> 62) == 2);
        const unsigned first = incl ? (unsigned)__ffs(incl) - 1 : 32u;
        uint64_t v = lane <= first ? (s & VAL) : 0;
#pragma unroll
        for (int d = 16; d; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
        excl += v;
        if (incl) break;
    }
    if (lane == 0) status[tile] = (2ull << 62) | ((excl + aggregate) & VAL);
    return excl;
}

// position of the n-th (0-based) set bit of a 32-bit word
__device__ __forceinline__ int nth_set_bit32(uint32_t m, int n) { return (int)__fns(m, 0, n + 1); }

}  // namespace spl
