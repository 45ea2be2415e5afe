"""GPU tests (-m gpu) of the beam cut's select, cut and rank machinery against plain numpy / Python references, on
constructed score sets at the edges where a radix select goes wrong.

`sorted(queue, key=score, reverse=True)[:beam]` under a tie policy is, on the device: the score dictionary
(dict_build_kernel / dict_rank_kernel, up to DICT_MAX distinct scores), the 11-bit radix select (sel_hist_kernel /
sel_pick_kernel), the tie split by key (select_ties_by_key), the cut kernels and the rank sort.  Covered here:

  1. spl_topk on a fresh context per case, the path (dictionary, or dictionary then radix) pinned and read back from
     the device with one-element probe cuts: 2047 / 2048 / 2049 distinct scores, a per-CTA dictionary table that spills, the dictionary skip after
     an overflow, key ranges of 0 to 64 bits built from adjacent doubles, +-DBL_MAX, +-5e-324 and +-0.0, k at 0, 1,
     n - 1, n, n + 1 and at both ends of tie groups, n = 8192 t +- 1 (the cut tile), and `det` keys that differ only in
     one word, in the top bit of a word or in the last digit;
  2. the distributed select of the key-sharded driver (spl_dtopk_*) over 1 to 8 contexts in this process, in lockstep,
     with uneven and empty shards and tie groups split across them, ranks from spl_count_less;
  3. spl_count_less against bisect over Python tuples;
  4. formulas built for those edges, level by level against the CPU oracle of formulas.

Untested here: the 8-bit LSD sort path for 2^30 or more survivors (OS_MAX_ITEMS) and the card-set-sharded driver's
threshold / tie calls (spl_gs_threshold, spl_gs_tie_*), whose inputs need a live solver."""
import bisect

import numpy as np
import pytest
import torch

import formula_oracle
import oracle
import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200 import Formula
from splendor_rl_gym_b200.sharded import SEL_BITS, Comm, CudaBackend, ShardedSolver, _bitlen, _radix_select
from test_gpu_formula import FIELDS, _vs_oracle

pytestmark = pytest.mark.gpu

DICT_MAX = 2048       # spl_kernels.cuh: most distinct scores the dictionary path handles
CUT_TILE = 32 * 256   # CUT_ITEMS * TILE: elements per tile of cut_kernel / cut_det_kernel
HI_MASK = (1 << 41) - 1
SIGN = np.uint64(1 << 63)
DBL_MAX = float(np.finfo(np.float64).max)


# ------------------------------------------------------------------ score sets
def _skey(sc):
    """the order-preserving image of each double as the device builds it (larger double <=> larger key, -0.0 == +0.0);
    used to construct score sets with an exact key range and to predict the select's path"""
    b = np.ascontiguousarray(sc, np.float64).view(np.uint64).copy()
    b[b == SIGN] = 0
    return np.where(b >> np.uint64(63) == 1, ~b, b | SIGN)


def _unkey(k):
    k = np.asarray(k, np.uint64)
    return np.where(k >> np.uint64(63) == 1, k & ~SIGN, ~k).view(np.float64)


#: (bitlen(max key - min key), where the keys sit): 'zero' straddles +-0.0 through the subnormals of both signs, 'one'
#: starts at 1.0, 'neg' at -1e300; 64 spans -DBL_MAX .. DBL_MAX
RANGES = [(0, 'zero'), (1, 'zero'), (1, 'one'), (10, 'zero'), (10, 'neg'), (11, 'one'), (11, 'zero'), (12, 'zero'),
          (12, 'neg'), (22, 'one'), (23, 'zero'), (33, 'neg'), (33, 'zero'), (53, 'one'), (63, 'zero'), (64, 'all')]


def _span(bits, where, n, rng, pool=300):
    """n >= 2 scores drawn from `pool` values whose keys span exactly `bits` bits, both ends present"""
    if bits == 0:
        sc = np.where(rng.integers(0, 2, n) == 1, -0.0, 0.0)  # +-0.0 only: one score
    else:
        if bits == 64:
            base = _skey([-DBL_MAX])[0]
            offs = rng.integers(0, _skey([DBL_MAX])[0] - base, size=pool, dtype=np.uint64, endpoint=True)
            offs[:2] = 0, _skey([DBL_MAX])[0] - base
        else:
            top = (1 << bits) - 1
            if where == 'zero':
                base = np.uint64((1 << 63) - (1 << (bits - 1)) if bits > 1 else 1 << 63)
            else:
                base = _skey([1.0 if where == 'one' else -1e300])[0]
            offs = rng.integers(0, top, size=max(2, min(pool, top + 1)), dtype=np.uint64, endpoint=True)
            offs[:2] = 0, top
        vals = _unkey(base + offs)
        if where == 'zero' and bits > 1:
            vals = np.concatenate([vals, [0.0, -0.0, 5e-324, -5e-324]])
        elif where == 'zero':
            vals = np.concatenate([vals, [-0.0]])
        sc = vals[rng.integers(0, len(vals), n)]
        sc[rng.choice(n, 2, replace=False)] = vals[:2]
    assert np.isfinite(sc).all()
    k = _skey(sc)
    assert _bitlen(int(k.max()) - int(k.min())) == bits
    return sc


def _groups(sc):
    """sizes of the tie groups, best score first"""
    return np.unique(_skey(sc), return_counts=True)[1][::-1]


def _k_edges(sc):
    """0, 1, n - 1, n, n + 1, and the k that end exactly at the first and at the last element of tie groups at even and
    odd positions of the score order"""
    n, c = len(sc), _groups(sc)
    cum = np.cumsum(c)
    ks = {0, 1, n - 1, n, n + 1}
    for g in {0, 1, len(c) // 2, len(c) // 2 + 1, len(c) - 2}:
        if 0 <= g < len(c):
            ks |= {int(cum[g] - c[g] + 1), int(cum[g])}
    return sorted(k for k in ks if k >= 0)


DET_KEYS = ('hi_eq', 'lo_eq', 'top', 'last')


def _det_keys(sc, pattern, rng):
    """(lo, hi) keys, unique inside every tie group (the det order is then total):
    hi_eq  one hi word (bit 40 set), the lo words differ anywhere
    lo_eq  one lo word (bit 63 set), the hi words differ
    top    lo bit 63 and hi bit 40 set on about half of the keys
    last   one hi word and the high bits of lo shared: ties are told apart in the lowest digits of lo"""
    n = len(sc)
    key = _skey(sc)
    o = np.lexsort((rng.permutation(n), key))
    s = key[o]
    start = np.r_[0, np.flatnonzero(s[1:] != s[:-1]) + 1]
    rank = np.empty(n, np.uint64)
    rank[o] = np.arange(n) - np.repeat(start, np.diff(np.r_[start, n]))  # random order inside the group
    u = np.uint64
    if pattern == 'hi_eq':
        hi = np.full(n, (1 << 40) | 0x5A5, u)
        lo = rng.integers(0, 1 << 40, n, dtype=u) << u(24) | rank
    elif pattern == 'lo_eq':
        lo = np.full(n, (1 << 63) | 0x1234, u)
        hi = rng.integers(0, 1 << 17, n, dtype=u) << u(24) | rank
    elif pattern == 'top':
        hi = rng.integers(0, 2, n, dtype=u) << u(40) | rng.integers(0, 4, n, dtype=u)
        lo = rng.integers(0, 2, n, dtype=u) << u(63) | rank
    else:
        hi = np.full(n, (1 << 32) | 1, u)
        lo = u(0xC0DE << 48) | rank
    assert int(hi.max()) <= HI_MASK
    return lo, hi


def _order(sc, lo, hi, tie):
    """sorted(range(n), key=score (, key), reverse=True): -0.0 == +0.0 as Python compares them; stable keeps arrival
    order among equal scores, det orders them by the 105-bit key (hi, lo), larger first"""
    c = np.asarray(sc, np.float64) + 0.0  # -0.0 + 0.0 == +0.0
    if tie == 'stable':
        return np.argsort(-c, kind='stable')
    return np.lexsort((lo, hi, c))[::-1]


# ------------------------------------------------------------------ 1. spl_topk with the path pinned
def _ceil(a, b):
    return -(-a // b)


class _Ctx:
    """A fresh context and the dictionary skip counter that run_dict_select keeps on it: after a cut with more than
    DICT_MAX distinct scores, the next three cuts go straight to the radix select.

    The path of a cut is read from the device with a probe, a cut of one element: it has nothing to select or sort, and
    its launches differ by exactly the dictionary's two kernels (dict_build + dict_rank) between a context that builds
    the dictionary and one that skips it.  A probe right after a cut therefore shows whether that cut overflowed the
    dictionary and fell back to the radix select, and probes between cuts show the skip counter counting down."""

    SKIP = 3

    def __init__(self, eng):
        self.eng, self.skip = eng, 0
        self.probe_dict = self.call(np.ones(1), 1)[1]  # launches of a probe that builds the dictionary

    def call(self, sc, k, tie='stable', lo=None, hi=None):
        """one spl_topk call == the numpy order, index for index -> (indices, kernel launches)"""
        n = len(sc)
        if lo is None:
            lo, hi = np.arange(n, dtype=np.uint64), np.zeros(n, np.uint64)
        eng = self.eng
        scores = torch.from_numpy(np.ascontiguousarray(sc, np.float64)).to(eng.tdev)
        keys = torch.from_numpy(np.stack([lo, hi], 1).view(np.int64)).to(eng.tdev)
        l0 = eng.launch_count()
        got = eng.topk(scores, keys, k, tie).cpu().numpy()
        launches = eng.launch_count() - l0
        want = _order(sc, lo, hi, tie)[:k]
        assert np.array_equal(got, want), (tie, n, k, self.skip)
        if n and k:
            if self.skip:
                self.skip -= 1
            elif len(np.unique(_skey(sc))) > DICT_MAX:
                self.skip = self.SKIP
        return got, launches

    def probe(self):
        """-> True when the context built the dictionary for the probe, asserted against the skip counter"""
        tried = self.skip == 0
        launches = self.call(np.ones(1), 1)[1]
        assert launches == self.probe_dict - 2 * (not tried), (launches, self.probe_dict, self.skip)
        return tried

    def topk(self, sc, k, tie='stable', lo=None, hi=None, path=None):
        """a checked spl_topk call -> the path it took ('dict' or 'radix'; None when there was nothing to cut), confirmed
        by a probe.  `path` pins it first: an overflowing cut arms the skip for 'radix', probes use it up for 'dict'."""
        n = len(sc)
        distinct = len(np.unique(_skey(sc)))
        if path == 'radix' and self.skip == 0 and distinct <= DICT_MAX:
            self.call(np.arange(DICT_MAX + 1, dtype=np.float64), DICT_MAX // 2)
            assert not self.probe()
        if path == 'dict':
            assert distinct <= DICT_MAX
            while self.skip:
                self.probe()
        took = ('dict' if self.skip == 0 and distinct <= DICT_MAX else 'radix') if n and k else None
        self.call(sc, k, tie, lo, hi)
        self.probe()
        assert path is None or took is None or took == path
        return took


@pytest.fixture
def fresh():
    made = []

    def make():
        made.append(S.Engine(0))
        return _Ctx(made[-1])
    yield make
    for e in made:
        e.close()


@pytest.mark.parametrize('distinct', [DICT_MAX - 1, DICT_MAX, DICT_MAX + 1])
@pytest.mark.parametrize('n', [CUT_TILE + 1, 3_000_000])
@pytest.mark.parametrize('tie', ['stable', 'det'])
def test_topk_dictionary_capacity(fresh, distinct, n, tie):
    """DICT_MAX distinct scores still take the dictionary, one more falls back to the radix select; at 3 M elements every
    CTA of dict_build_kernel meets more distinct scores than its 1 024-slot staging table holds and spills into the
    global table."""
    rng = np.random.default_rng(distinct * 7 + n)
    vals = rng.permutation(np.linspace(-1e3, 1e3, distinct))
    sc = vals[rng.integers(0, distinct, n)]
    sc[rng.choice(n, distinct, replace=False)] = vals
    lo, hi = _det_keys(sc, 'top', rng) if tie == 'det' else (None, None)
    c = _groups(sc)
    mid = len(c) // 2
    ks = [n // 3, int(c[:mid].sum()), int(c[:mid + 1].sum()) + 1] if n > CUT_TILE + 1 else _k_edges(sc)
    for k in ks:
        took = fresh().topk(sc, k, tie, lo, hi)
        assert took == (None if k == 0 else 'dict' if distinct <= DICT_MAX else 'radix'), k


@pytest.mark.parametrize('tie', ['stable', 'det'])
def test_topk_dictionary_skip_after_overflow(fresh, tie):
    """One cut that overflows the dictionary, then four with few distinct scores on the same context: all five exact, and
    only the fourth of those goes back to the dictionary.  The four keep one state, so that nothing is left to sort and
    their launches differ by the select alone: 6 radix passes of two kernels without the dictionary, its two kernels
    with it."""
    ctx = fresh()
    rng = np.random.default_rng(17)
    many = rng.normal(size=20_000) * 1e6
    ctx.call(many, 7_000, tie, *(_det_keys(many, 'hi_eq', rng) if tie == 'det' else (None, None)))
    launches = []
    for i in range(4):
        few = _span(64, 'all', 30_000 + i, rng, pool=40)
        launches.append(ctx.call(few, 1, tie, *(_det_keys(few, DET_KEYS[i], rng) if tie == 'det' else (None, None)))[1])
    radix = 2 * _ceil(64, SEL_BITS)
    assert launches[0] == launches[1] == launches[2] == launches[3] + radix - 2, launches
    assert ctx.probe()  # and the dictionary stays in use


@pytest.mark.parametrize('tie', ['stable', 'det'])
@pytest.mark.parametrize('bits,where', RANGES)
def test_topk_key_ranges(fresh, bits, where, tie):
    """Key ranges of 0 to 64 bits (up to 6 select passes, the last one narrower than 11 bits), on the dictionary path and
    on the radix path, n on both sides of a cut tile, k at every edge."""
    ctx = fresh()
    rng = np.random.default_rng(bits * 31 + len(where))
    for n in (CUT_TILE - 1, 3 * CUT_TILE + 1):
        sc = _span(bits, where, n, rng)
        lo, hi = _det_keys(sc, DET_KEYS[RANGES.index((bits, where)) % 4], rng) if tie == 'det' else (None, None)
        for k in _k_edges(sc):
            for path in ('dict', 'radix'):
                ctx.topk(sc, k, tie, lo, hi, path)
    for k in (0, 1, 2):
        for path in ('dict', 'radix'):
            ctx.topk(np.array([-0.0]), k, tie, path=path)


@pytest.mark.parametrize('pattern', DET_KEYS)
@pytest.mark.parametrize('n', [CUT_TILE + 1, 3 * CUT_TILE - 1])
def test_topk_det_keys(fresh, pattern, n):
    """det ties split by key on both paths: keys equal in one word, told apart by the top bit of a word (hi bit 40, lo bit
    63) or by the last digit, the threshold group cut at its first, middle and last element."""
    ctx = fresh()
    rng = np.random.default_rng(n + DET_KEYS.index(pattern))
    for pool in (12, 400):
        sc = _span(53, 'one', n, rng, pool=pool)
        lo, hi = _det_keys(sc, pattern, rng)
        c = _groups(sc)
        ks = set(_k_edges(sc))
        for g in (0, 1, len(c) // 2):
            ks.add(int(c[:g].sum() + c[g] // 2))
        for k in sorted(ks):
            for path in ('dict', 'radix'):
                ctx.topk(sc, k, 'det', lo, hi, path)


# ------------------------------------------------------------------ 2. distributed top-k over R contexts
class _LockstepSum:
    """Comm.all_reduce(SUM) for contexts that all live in this process: the sum of their histograms, written back into
    each one in place"""

    def all_reduce(self, hists, op):
        total = torch.stack([h.to(torch.int64) for h in hists]).sum(0)
        for h in hists:
            h.copy_(total.to(h.dtype))
        return hists


def _dtopk(backends, shards, sc, lo, hi, K, tie):
    """ShardedSolver._beam_cut's select, cut and ranks with every rank in this process, stepped in lockstep
    -> per rank (local indices of the survivors in local rank order, their global ranks)"""
    dev = backends[0].device
    u = [len(s) for s in shards]
    u_total = sum(u)
    live = []
    for b, s in zip(backends, shards):
        scores = torch.from_numpy(np.ascontiguousarray(sc[s])).to(dev)
        if tie == 'det':
            keys = torch.from_numpy(np.stack([lo[s], hi[s]], 1).view(np.int64)).to(dev)
        else:  # the synthetic arrival key: larger == earlier
            arr = torch.from_numpy(s).to(dev)
            keys = torch.stack([u_total - arr, torch.zeros_like(arr)], dim=1).contiguous()
        live.append((scores, keys, *b.dtopk_begin(scores, keys)))  # the key tensors stay alive until dtopk_cut
    smin = min(x[2] for x, n in zip(live, u) if n)
    smax = max(x[3] for x, n in zip(live, u) if n)
    keep_all, all_ties = u_total <= K, True
    comm = _LockstepSum()

    def select(word, top, init):
        _radix_select(comm, top, lambda shift, bits, first: [b.dtopk_hist(word, shift, bits, first, smin) for b in backends],
                      lambda shift, first: [b.dtopk_pick(word, shift, first, first and init, K) for b in backends])
    if not keep_all:
        for b in backends:
            b.dtopk_set([0, K, 0, u_total, 0, 0])
        select(0, _bitlen(smax - smin), True)
        states = [b.dtopk_get() for b in backends]
        assert all(st == states[0] for st in states)
        if states[0][1] < states[0][3]:
            all_ties = False
            for word, wbits in (((1, 41), (2, 64)) if tie == 'det' else ((2, _bitlen(u_total)),)):
                select(word, wbits, False)
    cuts = [b.dtopk_cut('det' if tie == 'det' else 'det_ordered', keep_all, all_ties, smin, smax, n) for b, n in zip(backends, u)]
    out = []
    for r, (b, (idx, y, kl, kh)) in enumerate(zip(backends, cuts)):
        grank = torch.arange(idx.shape[0], dtype=torch.int64, device=dev)
        for g, (_, y2, kl2, kh2) in enumerate(cuts):
            if g != r and idx.shape[0] and y2.shape[0]:
                b.count_less(3, False, (y, kl, kh), (y2, kl2, kh2), grank, True, True)
        out.append((idx.cpu().numpy(), grank.cpu().numpy()))
    return out


def _shards(n, R, tie, rng):
    """global indices per rank: uneven sizes, rank R // 2 empty from three ranks on; stable deals out blocks of the arrival
    order in turn (every shard ascending, as the driver's rounds leave them), det scatters the elements in any order"""
    live = [r for r in range(R) if R < 3 or r != R // 2]
    w = np.arange(1, len(live) + 1, dtype=np.float64) ** 2
    if tie == 'det':
        owner = np.array(live)[rng.choice(len(live), size=n, p=w / w.sum())]
        return [rng.permutation(np.flatnonzero(owner == r)) for r in range(R)]
    cuts = np.sort(rng.choice(np.arange(1, n), size=min(n - 1, 5 * len(live)), replace=False))
    blocks = np.split(np.arange(n), cuts)
    return [np.concatenate([np.zeros(0, np.int64)] + [blk for i, blk in enumerate(blocks) if live[i % len(live)] == r])
            for r in range(R)]


@pytest.fixture(scope='module')
def ranks():
    engs = [S.Engine(0) for _ in range(8)]
    yield [CudaBackend(e) for e in engs]
    for e in engs:
        e.close()


@pytest.mark.parametrize('tie', ['stable', 'det'])
@pytest.mark.parametrize('bits,where', [(0, 'zero'), (1, 'zero'), (11, 'one'), (12, 'zero'), (33, 'neg'), (53, 'one'),
                                        (63, 'zero'), (64, 'all')])
@pytest.mark.parametrize('R', [1, 2, 3, 8])
def test_dtopk_across_contexts(ranks, R, bits, where, tie):
    """spl_dtopk_* + spl_count_less over R contexts == the numpy order: each shard's survivors in local rank order, their
    global ranks at the elements' positions in the global order, and the ranks of all shards a permutation of 0..K-1."""
    rng = np.random.default_rng(R * 1000 + bits * 3 + (tie == 'det'))
    n = 2 * CUT_TILE + 3 + R
    sc = _span(bits, where, n, rng, pool=60)
    lo, hi = _det_keys(sc, DET_KEYS[bits % 4], rng) if tie == 'det' else (None, None)
    shards = _shards(n, R, tie, rng)
    sizes = sorted(map(len, shards))
    assert sum(sizes) == n and (sizes[0] == 0) == (R >= 3) and len(set(sizes)) == R
    order = _order(sc, lo, hi, tie)
    for K in _k_edges(sc):
        if K == 0:
            continue
        out = _dtopk(ranks[:R], shards, sc, lo, hi, K, tie)
        top = order[:min(K, n)]
        pos = np.full(n, -1)
        pos[top] = np.arange(len(top))
        got = []
        for (idx, grank), s in zip(out, shards):
            mine = s[pos[s] >= 0]
            mine = mine[np.argsort(pos[mine])]
            assert np.array_equal(s[idx], mine), (K, len(s))
            assert np.array_equal(grank, pos[mine]), (K, len(s))
            got.append(grank)
        assert np.array_equal(np.sort(np.concatenate(got)), np.arange(len(top))), K


# ------------------------------------------------------------------ 3. spl_count_less
def _u64(x):
    return torch.from_numpy(np.asarray(x, np.uint64).view(np.int64))


@pytest.mark.parametrize('sorted_a', [0, 1])
@pytest.mark.parametrize('accumulate', [0, 1])
@pytest.mark.parametrize('inclusive', [0, 1])
@pytest.mark.parametrize('words', [1, 3])
def test_count_less(ranks, words, inclusive, accumulate, sorted_a):
    """out[i] (+)= #{j: b[j] < a[i]} (<= when inclusive) for composites (y, kh, kl) compared as unsigned words ==
    bisect over Python tuples: equal y told apart by kh or only by kl, duplicates of a inside b, empty a or b, lengths
    at the 256-thread tile edges."""
    b_ = ranks[0]
    dev = b_.device
    rng = np.random.default_rng(words * 8 + inclusive * 4 + accumulate * 2 + sorted_a)
    ys = [0, 1, 5, (1 << 63) - 1, 1 << 63, (1 << 64) - 1]
    ks = [0, 2, 1 << 40, (1 << 63) + 9, (1 << 64) - 2]
    rand = lambda m: [(ys[rng.integers(len(ys))], ks[rng.integers(len(ks))], ks[rng.integers(len(ks))]) for _ in range(m)]  # noqa: E731
    for na, nb in [(0, 50), (50, 0), (255, 256), (256, 257), (257, 255), (1, 1), (513, 1024), (4097, 3000)]:
        b = sorted(rand(nb))
        a = rand(na - na // 2) + [b[i] for i in rng.integers(0, max(nb, 1), na // 2)] if nb else rand(na)
        a = sorted(a) if sorted_a else [a[i] for i in rng.permutation(na)]
        cut = (lambda t: t) if words == 3 else (lambda t: t[:1])
        bt = [cut(t) for t in b]
        r = [(bisect.bisect_right if inclusive else bisect.bisect_left)(bt, cut(t)) for t in a]
        prev = rng.integers(-1000, 1000, na)
        col = lambda ts, j: _u64([t[j] for t in ts]).to(dev)  # noqa: E731
        A = (col(a, 0), col(a, 2), col(a, 1))  # (y, kl, kh)
        B = (col(b, 0), col(b, 2), col(b, 1))
        out = torch.from_numpy(prev.copy()).to(dev)
        b_.count_less(words, inclusive, A, B, out, accumulate, sorted_a)
        want = np.asarray(r, np.int64) + (prev if accumulate else 0)
        assert np.array_equal(out.cpu().numpy(), want), (na, nb)


# ------------------------------------------------------------------ 4. formulas built for the cut's edges
#: terms near the finiteness bound with both signs: every noise draw vanishes, ties are massive and the key range spans
#: 64 bits; a zero exponent (x ** 0.0 == 1, also at x == 0)
HUGE = Formula([(5e305, ('pts', 1.0)), (-3e305, ('gem_red', 1.0), ('gem_blue', 0.0)), (-1e305, ('cards', 1.0))])
#: a subnormal coefficient and one near the subnormals: both terms are subnormal numbers on queued states (they vanish
#: once the larger terms and the noise term are added)
TINY = Formula([(5e-324, ('saved', 1.0)), (-2.5e-310, ('gems', 1.5), ('colors', 0.0)), (1.0, ('pts', 2.0)),
                (-0.75, ('cards', 1.0))])
#: thousands of distinct scores per level at beam 20 000: the dictionary overflows on the later levels
WIDE = Formula([(25.0, ('pts', 2.05)), (1e-2, ('gem_white', 1.1), ('bonus_white', 0.7)), (-1e-3, ('gem_blue', 1.3), ('saved', 0.45)),
                (1e-4, ('gem_green', 1.7)), (-1e-5, ('gem_red', 0.6), ('bonus_red', 1.9)), (1e-6, ('gem_black', 2.3), ('cards', 1.1)),
                (-3e-8, ('bonus', 1.5), ('gem_white', 0.0))])
EDGE = {'huge': HUGE, 'tiny': TINY, 'wide': WIDE}


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


@pytest.fixture(scope='module')
def edge_levels():
    """per formula: (states, scores with noise const) of every queue after a cut of the oracle's search at beam 20 000"""
    out = {}
    for name, f in EDGE.items():
        orc = formula_oracle.Solver(15, f, beam_width=20_000)
        orc.run()
        out[name] = [(st, formula_oracle.score(st, f)) for st in (orc.level(i)[0] for i in range(1, len(orc.infos)))]
        orc.close()
    return out


def test_edge_formulas_reach_their_edges(edge_levels):
    """the premises of the formulas above hold on the queues of their searches"""
    def span(sc):
        k = _skey(sc)
        return _bitlen(int(k.max()) - int(k.min()))
    huge, tiny, wide = edge_levels['huge'], edge_levels['tiny'], edge_levels['wide']
    assert any((sc < 0).any() and (sc > 0).any() and span(sc) == 64 for _, sc in huge)
    assert max(len(sc) for _, sc in huge) == 20_000 and max(len(np.unique(sc)) for _, sc in huge) <= 64  # massive ties
    assert max(len(np.unique(sc)) for _, sc in wide) > DICT_MAX  # (the unique states of such a level, a superset, too)
    assert any((sc < 0).any() and (sc > 0).any() for _, sc in tiny)
    st = np.concatenate([s for s, _ in tiny])
    saved = (st['aux'] & np.uint64(0xffff)).astype(np.float64)
    gems = sum((st['lo'] >> np.uint64(3 * c)) & np.uint64(7) for c in range(5)).astype(np.float64)
    for t in (5e-324 * saved, -2.5e-310 * gems ** 1.5):  # the first two terms of TINY
        assert ((t != 0) & (np.abs(t) < np.finfo(np.float64).tiny)).any()


@pytest.mark.parametrize('name,noise', [('huge', 'const'), ('tiny', 'hash'), ('wide', 'const'), ('wide', 'hash')])
def test_edge_formulas_grouped_level(eng, name, noise):
    _vs_oracle(eng, EDGE[name], 20_000, noise=noise)


@pytest.mark.parametrize('name,beam,noise', [('huge', 5_000, 'hash'), ('tiny', 5_000, 'const'), ('wide', 20_000, 'hash')])
def test_edge_formulas_key_table_level_det(eng, name, beam, noise, monkeypatch):
    monkeypatch.setenv('SPL_NO_GROUPED', '1')
    _vs_oracle(eng, EDGE[name], beam, policy='det', noise=noise)


@pytest.mark.parametrize('name,tie,noise', [('huge', 'stable', 'const'), ('tiny', 'det', 'hash'), ('wide', 'stable', 'hash'),
                                            ('wide', 'det', 'const')])
def test_edge_formulas_sharded_world1(eng, name, tie, noise):
    """the key-sharded driver at world 1 (every cut through spl_dtopk_* and the radix select) against the oracle"""
    f, beam = EDGE[name], 20_000
    sol = ShardedSolver(CudaBackend(eng), Comm(eng.tdev), 0, 0, 15, True, f, beam, tie, noise, block_parents=1 << 14)
    orc = formula_oracle.Solver(15, f, beam_width=beam, policy=tie, noise=noise)
    try:
        while True:
            gi, oi = sol.step(), orc.step()
            fields = ('frontier', 'goal_rank') if gi['ended'] else FIELDS
            assert {x: gi[x] for x in fields} == {x: oi[x] for x in fields}, (name, gi, oi)
            if gi['ended']:
                break
            fr = sol.gather_frontier().cpu().numpy().view(np.uint64)
            st, lk = orc.level(oi['level'] + 1)
            assert fr.tobytes() == np.stack([st['lo'], st['hi'], st['aux'], lk], 1).tobytes(), (name, gi['level'])
        ords = sol.path()[1]
        want = orc.path()
        line = [want[:1].copy()]
        for o in ords:
            line.append(oracle.expand(line[-1])[o:o + 1])
        assert np.concatenate(line).tobytes() == want.tobytes(), name
    finally:
        orc.close()
        eng.reset_visited()
