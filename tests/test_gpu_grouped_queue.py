"""The single-GPU grouped level (csrc/spl_m2.cuh, ordered instantiations) on level-0 queues built on purpose (-m gpu).

spl_solver_create_queue starts the solver from chosen rows, so a test picks the round's parents: buyers T \\ {c} of a
target card set T (tests/grouped_ref.py `buyer`) put buy items under chosen sort keys, at chosen item indices
(np + boff[p] + ordinal) and in chosen rounds, and filler rows (no bonus, no gems: no buys, 15 takes) set a round's
item count exactly.  Buys travel as 8-byte sort items and are rebuilt from their parents' records (load_buy), and the
first arrival of a state relies on the stable item sort alone.  Every level is compared with the host reference
(full rows {lo, hi, aux, link}, `unique`, `visited`, `kept`), and every round's `[grouped]` line (SPL_DEBUG) must show
the items, runs and run classes the host predicts with the single-GPU threshold BIG_W, so each test shows that it
reached the kernel it is about."""
import re

import numpy as np
import pytest

import grouped_ref as G
import oracle
import splendor_rl_gym_b200 as S

pytestmark = pytest.mark.gpu

LINE = re.compile(r'\[grouped\] L(\d+) np=(\d+) items=(\d+) runs=(\d+) cls=(\d+)/(\d+)/(\d+) ')
SHIFT = G.SORT_SHIFT


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def _lines(capfd):
    return [tuple(int(x) for x in m.groups()) for m in LINE.finditer(capfd.readouterr().err)]


def _front(sol):
    return np.ascontiguousarray(sol.frontier().cpu().numpy()).view(G.REC_DTYPE).reshape(-1)


def _key(r):
    return int(r['lo']), int(r['hi'])


class Run:
    """The single-GPU solver started from a constructed queue, stepped beside G.ref_level."""

    def __init__(self, eng, capfd, rows, heuristic='simple', beam=10 ** 7, chunk=None):
        self.queue = G.queue_of(rows)
        self.capfd, self.heuristic, self.beam = capfd, heuristic, beam
        self.chunk = chunk or 16 << 20  # the Engine's chunk_parents (default: MAX_CHUNK_PARENTS)
        self.visited = {_key(r) for r in self.queue}
        self.sol = eng.solver(0, 0, 255, True, heuristic, beam, queue=self.queue)

    def step(self):
        """one level; returns (next queue, [per round: (items, {sort key: (class, sets, items, candidates)})])"""
        gi = self.sol.step()
        lines = _lines(self.capfd)
        cands, ntk = G.expand_queue(self.queue)
        nxt, unique = G.ref_level(self.queue, self.visited, None, self.heuristic, beam=self.beam, expanded=cands)
        assert (gi['unique'], gi['visited'], gi['kept']) == (unique, len(self.visited), len(nxt)), gi
        assert np.array_equal(_front(self.sol), nxt)
        par = (cands['link'] >> np.uint64(8)).astype(np.int64)
        n = len(self.queue)
        assert len(lines) == -(-n // self.chunk)
        rounds = []
        for r, line in enumerate(lines):
            lo, hi = r * self.chunk, min(n, (r + 1) * self.chunk)
            buys = G.buys_of(self.queue, cands[(par >= lo) & (par < hi)])
            n_runs, cls, runs = G.predict_runs(self.queue[lo:hi], ntk[lo:hi], buys, warp_max=G.WARP_MAX_ORDERED)
            assert line[1:7] == (hi - lo, hi - lo + len(buys), n_runs) + cls, (r, line, n_runs, cls)
            rounds.append((hi - lo + len(buys), runs))
        self.queue = nxt
        return nxt, rounds

    def close(self):
        self.sol.close()


def _winner(nxt, m0, m1, gems):
    key = G.make_row(m0, m1, gems)
    hit = nxt[(nxt['lo'] == np.uint64(key[0])) & (nxt['hi'] == np.uint64(key[1]))]
    assert len(hit) == 1
    return int(hit['link'][0]) >> 8, int(hit['link'][0]) & 0xff


def _sets_under(rng, k, n, twin=True, m1_or=0):
    """n card sets under sort key k; with `twin` the first two have the same 64-bit hash"""
    out = []
    for i in range(n):
        h = out[0][2] if (twin and i == 1) else k << SHIFT | int(rng.integers(0, 1 << SHIFT))
        m1 = int(rng.integers(0, 1 << 26)) | m1_or
        out.append((G.m0_for_hash(h, m1), m1, h))
    assert len({(a, b) for a, b, _ in out}) == n and all(G.sort_key(G.hash_key(a, b)) == k for a, b, _ in out)
    return [(a, b) for a, b, _ in out]


def _fresh_keys(rng, n):
    return [int(x) for x in rng.choice(np.arange(1, 1 << 20, dtype=np.int64), n, replace=False) << 10 | rng.integers(0, 1 << 10, n)]


def _buyers(rng, T, n, hands, skip=()):
    """n buyers of card set T: distinct (missing card, hand) pairs, hands cycled"""
    cards = [c for c in G.cards_of(*T) if c not in skip]
    rng.shuffle(cards)
    out = []
    for j in range(n):
        out.append(G.buyer(*T, cards[j % len(cards)], hands[(j // len(cards) + j % len(cards)) % len(hands)]))
    assert len(set(r[:2] for r in out)) == n
    return out


def _fillers(rng, n, taken=()):
    rows, seen = [], set(taken)
    while len(rows) < n:
        m = int(rng.integers(1, 1 << 62)), int(rng.integers(0, 1 << 26))
        if m not in seen:
            seen.add(m)
            rows.append(G.filler(*m))
    return rows


HANDS = [(1, 1, 1, 0, 0), (0, 1, 1, 1, 0), (2, 0, 0, 1, 1), (0, 0, 0, 0, 0), (1, 0, 2, 0, 1)]


# ------------------------------------------------------------------ 1. a queue start against the oracle
def _oracle_queue(seed, n, pts):
    rng = np.random.default_rng(seed)
    rows, seen = [], set()
    while len(rows) < n:
        cards = rng.choice(90, int(rng.integers(0, 9)), replace=False).tolist()
        g = G.random_hand(rng)
        if sum(g) > 6:
            continue
        r = G.make_row(*G.card_set(cards), g, tuple(int(x) for x in rng.integers(0, 4, 5)), int(rng.integers(*pts)),
                       int(rng.integers(0, 20)))
        if r[:2] not in seen:
            seen.add(r[:2])
            rows.append(r)
    return G.queue_of(rows)


def _levels_equal_oracle(sol, orc, max_levels=None):
    lv = 0
    while True:
        gi, oi = sol.step(), orc.step()
        for f in ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'generated', 'unique', 'kept', 'visited'):
            assert gi[f] == oi[f], (lv, f, gi, oi)
        if gi['ended']:
            return True
        st, lk = orc.level(lv + 1)
        fr = _front(sol)
        assert (fr['lo'] == st['lo']).all() and (fr['hi'] == st['hi']).all() and (fr['aux'] == st['aux']).all()
        assert (fr['link'] == lk).all()
        lv += 1
        if max_levels and lv >= max_levels:
            return False


@pytest.mark.parametrize('hname', ['simple', 'aggressive'])
@pytest.mark.parametrize('beam,levels', [(2000, None), (10 ** 7, 2)])
@pytest.mark.parametrize('grouped', [True, False])
def test_queue_start_equals_oracle(eng, monkeypatch, hname, beam, levels, grouped):
    """A 1500-row queue run to the goal with beam 2000, or two levels with no cut: every level equals the oracle's
    restatement started from the same rows, and so does the path; with SPL_NO_GROUPED=1 the key-table level gives the
    same levels from the same create."""
    if not grouped:
        monkeypatch.setenv('SPL_NO_GROUPED', '1')
    q = _oracle_queue(7 + beam, 1500, (6, 12) if levels is None else (0, 5))  # the goal within reach / out of reach
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name=hname, beam_width=beam, root=q)
    sol = eng.solver(0, 0, 15, True, hname, beam, queue=q)
    try:
        assert np.array_equal(orc.level(0)[0]['lo'], q['lo'])
        ended = _levels_equal_oracle(sol, orc, levels)
        assert ended == (levels is None)
        if ended:
            ranks, ords = sol.path()
            want = orc.path()
            assert len(ranks) == len(want) >= 2
            for l, r in enumerate(ranks):
                st, _ = orc.level(l)
                assert _key(st[r]) == _key(want[l]) and st['aux'][r] == want['aux'][l]
            for l, o in enumerate(ords):
                assert _key(oracle.expand(want[l:l + 1])[o]) == _key(want[l + 1])
    finally:
        sol.close()
        orc.close()


def test_one_row_queue_equals_create():
    """A queue of the new-game root alone is spl_solver_create: the same levels, launches and host<->device bytes
    (each on a fresh Engine, so that neither solve finds tables grown by the other)."""
    k, a = S.State.newgame().record()
    q = G.queue_of([(k & G.M64, k >> 64, a, 0)])
    out = []
    for queue in (None, q):
        eng = S.Engine(0)
        l0, t0 = eng.launch_count(), eng.transfer_bytes()
        sol = eng.solver(k, a, 15, True, 'aggressive', 3000, queue=queue)
        infos = [{f: v for f, v in sol.step().items() if not f.startswith('ms_')} for _ in range(6)]
        l1, t1 = eng.launch_count(), eng.transfer_bytes()
        out.append((infos, l1 - l0, (t1[0] - t0[0], t1[1] - t0[1]), _front(sol).copy()))
        sol.close()
        eng.close()
    assert out[0][:3] == out[1][:3]
    assert np.array_equal(out[0][3], out[1][3])


# ------------------------------------------------------------------ 2. several card sets under one sort key
def _shared_key_queue(seed):
    """level-0 rows and {sort key: (class, sets)}: 2..5 sets under one key as a tiny-sized buy-only run and as a warp
    run, 17 sets as a CTA run (the first two sets of each with one 64-bit hash); a parent run whose key also holds
    two sets reached only by buys of other parents; and, for every target set, a row T \\ {c'} with no gems whose
    take child at level 1 buys c' into (T, hand) again at level 2"""
    rng = np.random.default_rng(seed)
    keys = iter(_fresh_keys(rng, 16))
    rows, want, again, targets = [], {}, [], []
    for n in (2, 3, 4, 5):
        for cls, per_set in ((G.WARP, 2), (G.WARP, 9)):
            k = next(keys)
            for T in _sets_under(rng, k, n):
                rows += _buyers(rng, T, per_set, HANDS[:3], skip=G.cards_of(*T)[:1])
                targets.append(T)
            want[k] = (cls, n)
    k = next(keys)
    for T in _sets_under(rng, k, 17):
        rows += _buyers(rng, T, 61, HANDS[:3], skip=G.cards_of(*T)[:1])
        targets.append(T)
    want[k] = (G.CTA, 17)
    k = next(keys)
    P, *others = _sets_under(rng, k, 3)
    rows += [G.make_row(*P, g) for g in HANDS]                       # the parents of the run: 5 hands, their takes
    for T in others:
        rows += _buyers(rng, T, 4, HANDS[:2])
        targets.append(T)
    want[k] = (G.WARP, 3)
    for T in targets:  # (T \ {c'}, no gems) takes (1, 1, 1, 0, 0) and buys c' one level later
        c = G.cards_of(*T)[0]
        again.append(G.buyer(*T, c, (0,) * 5))
    perm = rng.permutation(len(rows))
    rows = [rows[i] for i in perm]
    return rows + again, want, targets


def test_shared_sort_keys(eng, capfd, monkeypatch):
    monkeypatch.setenv('SPL_DEBUG', '1')
    rows, want, targets = _shared_key_queue(11)
    run = Run(eng, capfd, rows)
    try:
        nxt, rounds = run.step()
        runs = rounds[0][1]
        for k, (cls, n) in want.items():
            assert runs[k][:2] == (cls, n), (k, runs[k], cls, n)
        assert runs[min(want, key=lambda k: (want[k][0] != G.WARP, want[k][1]))][2] <= G.TINY_ITEMS
        won = {_key(r) for r in nxt}
        again = {G.make_row(*T, (1, 1, 1, 0, 0))[:2] for T in targets}
        assert again <= won  # every target set won hand (1, 1, 1, 0, 0) at level 1 ...
        visited = set(run.visited)
        cands, _ = G.expand_queue(nxt)
        assert again <= {_key(r) for r in cands}  # ... and reaches it again at level 2
        nxt2, _ = run.step()
        assert not again & {_key(r) for r in nxt2} and again <= visited
    finally:
        run.close()


# ------------------------------------------------------------------ 3. limits
@pytest.mark.parametrize('n_sets,per_set,cls', [(6, 4, G.WARP), (18, 61, G.CTA)])
def test_too_many_sets_under_one_sort_key(eng, capfd, monkeypatch, n_sets, per_set, cls):
    """One more card set under a sort key than the kernel of its class walks: the level fails and says so; the Engine
    then runs a normal search that equals the oracle."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    rng = np.random.default_rng(21 + n_sets)
    k = _fresh_keys(rng, 1)[0]
    rows = []
    for T in _sets_under(rng, k, n_sets):
        rows += _buyers(rng, T, per_set, HANDS[:3])
    q = G.queue_of(rows)
    sol = eng.solver(0, 0, 255, True, 'simple', 10 ** 7, queue=q)
    try:
        with pytest.raises(S.SplendorB200Error, match='more than 5 card sets share one 30-bit sort key .* more than 17 '):
            sol.step()
    finally:
        sol.close()
    cands, ntk = G.expand_queue(q)
    n_runs, counts, runs = G.predict_runs(q, ntk, G.buys_of(q, cands), warp_max=G.WARP_MAX_ORDERED)
    lines = _lines(capfd)
    assert len(lines) == 1 and lines[0][3:7] == (n_runs,) + counts and runs[k][:2] == (cls, n_sets)
    monkeypatch.delenv('SPL_DEBUG')
    k0, a0 = S.State.newgame().record()
    sol = eng.solver(k0, a0, 15, True, 'aggressive', 5000, 'stable', 'const')
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name='aggressive', beam_width=5000)
    try:
        assert _levels_equal_oracle(sol, orc)
    finally:
        sol.close()
        orc.close()


# ------------------------------------------------------------------ 4. first arrival across parents, class edges
def _hand(row):
    return tuple(int(row[0]) >> (3 * i) & 7 for i in range(5))


def _take_hands(gems):
    """the hands of the gem-take successors of a row with hand `gems` (takes depend on the hand alone)"""
    q = G.queue_of([G.make_row(*G.card_set([0]), gems)])
    cands = G.expand_queue(q)[0]
    same = cands[(cands['lo'] >> np.uint64(15) == q['lo'][0] >> np.uint64(15)) & (cands['hi'] == q['hi'][0])]
    return [_hand(r) for r in same]


def _ntk(gems):
    return len(_take_hands(gems))


@pytest.mark.parametrize('weight', [1024, 1025])
def test_class_edges_and_first_arrival(eng, capfd, monkeypatch, weight):
    """Buy-only runs of one card set with 16 and 17 items (thread / warp kernel) whose buyers share hands; a parent
    run of `weight` candidates (warp kernel up to BIG_W = 1024, CTA kernel beyond) made of its parents' takes and
    buys whose hands equal those takes, from buyers ranked before, between and after the parents; and the warp
    kernel's paired step: two parents of one set with at most 16 takes each and a buy from a row ranked between them
    that shares a take hand of the second."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    rng = np.random.default_rng(weight)
    k16, k17, kw, kp = _fresh_keys(rng, 4)
    want = {}
    head = []
    for k, n, cls in ((k16, 16, G.THREAD), (k17, 17, G.WARP)):
        T = _sets_under(rng, k, 1)[0]
        head += _buyers(rng, T, n, HANDS[:2])
        want[k] = (cls, 1, n, n)
    # the heavy parent run: parents of P with hands of known take counts, buyers of P filling the weight exactly
    P = _sets_under(rng, kw, 1)[0]
    par_hands = [(3, 3, 3, 1, 0), (2, 2, 2, 2, 2), (1, 1, 1, 0, 0), (0, 0, 0, 0, 0), (7, 3, 0, 0, 0)]
    parents = [G.make_row(*P, g) for g in par_hands]
    w = sum(_ntk(g) for g in par_hands)
    takes = _take_hands((2, 2, 2, 2, 2))
    n_buy = weight - w
    cards = G.cards_of(*P)
    hands = [h for h in takes if h not in par_hands]
    buys = [G.buyer(*P, cards[j % len(cards)], hands[j // len(cards)]) for j in range(n_buy)]
    assert len(set(r[:2] for r in buys)) == n_buy
    want[kw] = (G.WARP if weight <= G.WARP_MAX_ORDERED else G.CTA, 1, len(parents) + n_buy, weight)
    # the paired step: parents (Q, a) .. (Q, b) with <= 16 takes, a buyer of (Q, take of b) between them
    Q = _sets_under(rng, kp, 1)[0]
    qa, qb = (0, 0, 0, 0, 0), (1, 0, 0, 0, 0)
    assert _ntk(qa) <= 16 and _ntk(qb) <= 16
    shared = [h for h in _take_hands(qb) if h not in _take_hands(qa)][0]
    pair = [G.make_row(*Q, qa), G.buyer(*Q, G.cards_of(*Q)[-1], shared), G.make_row(*Q, qb)]
    rows = buys[:n_buy // 3] + head + parents[:3] + buys[n_buy // 3: 2 * n_buy // 3] + parents[3:] + pair + \
        buys[2 * n_buy // 3:]
    run = Run(eng, capfd, rows)
    try:
        nxt, rounds = run.step()
        runs = rounds[0][1]
        for k, wnt in want.items():
            assert runs[k] == wnt, (k, runs[k], wnt)
        assert runs[kp][0] == G.WARP
        rank = {r[:2]: i for i, r in enumerate(rows)}
        # the buyer between the pair beats the second parent's take
        assert _winner(nxt, *Q, shared)[0] == rank[pair[1][:2]]
        # hands of P that a buy and a take both reach: the first arrival wins, a buy before a take and the reverse
        par_rank = {rank[r[:2]]: set(_take_hands(_hand(r))) for r in parents}
        buy_first = take_first = 0
        for b in buys:
            g, rb = _hand(b), rank[b[:2]]
            takers = [p for p, hs in par_rank.items() if g in hs]
            if takers:
                w = _winner(nxt, *P, g)[0]
                assert w == min([rb] + takers + [rank[x[:2]] for x in buys if _hand(x) == g])
                buy_first += w == rb and rb < min(takers)
                take_first += w in takers and rb > w
        assert buy_first and take_first
    finally:
        run.close()


# ------------------------------------------------------------------ 5. sort stability
def _spacer(i, g):
    """a one-card row that can afford every other card: 89 buy items"""
    return G.make_row(*G.card_set([i]), g, (7,) * 5)


@pytest.mark.parametrize('n_items', [1, 4095, 4096, 4097, 8192, 8193])
def test_sort_stability(eng, capfd, monkeypatch, n_items):
    """Pairs of buyers of one target set with one hand: both children are one state, and only the lower-ranked
    buyer's copy may win.  The copies' item indices np + boff[p] + ordinal lie in one warp's 512 items, in two warps
    of one 4096-item tile, in two tiles, and in the last partial tile (the very last item); fillers make the round
    exactly n_items items."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    rng = np.random.default_rng(n_items)
    if n_items == 1:
        run = Run(eng, capfd, _fillers(rng, 1))
        try:
            assert run.step()[1][0][0] == 1
        finally:
            run.close()
        return
    spacers = iter([_spacer(i, g) for g in HANDS for i in range(90)])
    layout = [('warp', 0), ('tile', 6)] + ([('cross', 48)] if n_items >= 2 * G.SORT_TILE else [])
    if n_items % G.SORT_TILE and n_items > G.SORT_TILE:
        layout.append(('last', 0))
    rows, pairs = [], []
    for name, gap in layout:
        T = _sets_under(rng, _fresh_keys(rng, 1)[0], 1, m1_or=1 << 25)[0]  # card 89 in T: its buy is a buyer's last
        c0 = G.cards_of(*T)[0]
        a, b = G.buyer(*T, c0, HANDS[0]), G.buyer(*T, 89, HANDS[0])
        rows += [a] + [next(spacers) for _ in range(gap)] + [b]
        pairs.append((name, T, (a, c0), (b, 89)))
    q = G.queue_of(rows)
    n_buys = len(G.buys_of(q, G.expand_queue(q)[0]))
    assert n_items - n_buys >= len(rows)
    rows += _fillers(rng, n_items - n_buys - len(rows))
    q = G.queue_of(rows)
    buys = G.buys_of(q, G.expand_queue(q)[0])
    par = (buys['link'] >> np.uint64(8)).astype(np.int64)
    assert len(q) + len(buys) == n_items
    rank = {r[:2]: i for i, r in enumerate(rows)}

    def item(row, card):
        """np + boff[p] + ordinal of row's buy of `card`"""
        p = rank[row[:2]]
        m0, m1 = G.card_words_np(buys['lo'], buys['hi'])
        has = (m0 >> np.uint64(card) & np.uint64(1)) if card < 64 else (m1 >> np.uint64(card - 64) & np.uint64(1))
        hit = np.nonzero((par == p) & (has == 1))[0]
        assert len(hit) == 1
        return len(q) + int(hit[0])
    for name, T, (a, ca), (b, cb) in pairs:
        ia, ib = item(a, ca), item(b, cb)
        wa, wb, ta, tb = ia // G.SORT_ITEMS_WARP, ib // G.SORT_ITEMS_WARP, ia // G.SORT_TILE, ib // G.SORT_TILE
        if name == 'warp':
            assert wa == wb, (name, ia, ib)
        elif name == 'tile':
            assert ta == tb and wa != wb, (name, ia, ib)
        elif name == 'cross':
            assert ta != tb, (name, ia, ib)
        else:
            assert ib == n_items - 1 and ta != tb, (name, ia, ib)
    run = Run(eng, capfd, rows)
    try:
        nxt, rounds = run.step()
        assert rounds[0][0] == n_items
        for name, T, (a, _), _ in pairs:
            assert _winner(nxt, *T, HANDS[0])[0] == rank[a[:2]], name
    finally:
        run.close()


# ------------------------------------------------------------------ 6. rebuilt buys at the key's word edges
def test_rebuilt_buys_at_word_edges(eng, capfd, monkeypatch):
    """Buyers lacking card 0, 48, 49 or 89 (key bits 15, 63, 64, 104) whose bonus is below the card's cost, so that
    the buy pays part in gems: child keys, saved gems, points, bonus and link ordinals equal oracle.expand's; the
    buys of cards 49 and 89 come after buys of lower cards (their ordinals count the low word)."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    rng = np.random.default_rng(6)
    rows, missing = [], []
    for c in (0, 48, 49, 89):
        cost = G.card_cost(c)
        bonus = tuple(max(x - 1, 0) for x in cost)
        for extra in ((0, 0, 0, 0, 0), (1, 1, 0, 0, 0), (0, 0, 2, 1, 0)):
            gems = tuple(min(7, (1 if x else 0) + e) for x, e in zip(cost, extra))
            for _ in range(2):
                m = int(rng.integers(0, 1 << 63)) | int(rng.integers(0, 1 << 26)) << 64 | 1 << c
                T = (m & G.M64, m >> 64)
                rows.append(G.buyer(*T, c, gems, bonus, pts=int(rng.integers(0, 9)), saved=int(rng.integers(0, 50))))
                missing.append(c)
    q = G.queue_of(rows)
    cands, _ = G.expand_queue(q)
    paid = 0
    for p, (r, c) in enumerate(zip(rows, missing)):
        kids = cands[cands['link'] >> np.uint64(8) == np.uint64(p)]
        kid = [k for k in kids if (int(k['lo']) >> 15 | int(k['hi']) << 49) >> c & 1][0]
        paid += (int(kid['lo']) & 0x7FFF) != (r[0] & 0x7FFF)
        if c in (49, 89):
            assert int(kid['link']) & 0xff > 0
    assert paid == len(rows)
    run = Run(eng, capfd, rows, 'aggressive')
    try:
        nxt, _ = run.step()
        run.step()
    finally:
        run.close()


# ------------------------------------------------------------------ 7. several rounds per level
def test_rounds_carry_rank_base(capfd, monkeypatch):
    """Rounds of 256 parents: buyers of one target set whose hands repeat across rounds, so that the first arrival of
    a state lies in an earlier round than its copies; links carry rank_base + p."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    eng2 = S.Engine(0, chunk_parents=256)
    rng = np.random.default_rng(7)
    T = _sets_under(rng, _fresh_keys(rng, 1)[0], 1)[0]
    cards = G.cards_of(*T)
    rows = _fillers(rng, 1000)
    slots = sorted(rng.choice(1000, 24, replace=False).tolist())
    for j, s in enumerate(slots):
        rows[s] = G.buyer(*T, cards[j], HANDS[j % 3])
    run = Run(eng2, capfd, rows, chunk=256)
    try:
        nxt, rounds = run.step()
        assert len(rounds) == 4
        for h in range(3):
            assert _winner(nxt, *T, HANDS[h])[0] == slots[h]
        assert max(int(r['link']) >> 8 for r in nxt) >= 768
        run.step()
    finally:
        run.close()
        eng2.close()


# ------------------------------------------------------------------ 8. rejected rows
def test_rejected_rows(eng, capfd, monkeypatch):
    """An illegal gem hand, a key bit at or above 105 and a second row with one key are rejected on the host, naming
    the row; the context runs a queue afterwards."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    rng = np.random.default_rng(8)
    good = _fillers(rng, 3)
    bad_hand = list(good[1])
    bad_hand[0] = (bad_hand[0] & ~0x7FFF) | 3 | 3 << 3 | 3 << 6 | 2 << 9  # 11 gems
    bad_bit = list(good[1])
    bad_bit[1] |= 1 << 41
    for rows, msg in (([good[0], tuple(bad_hand), good[2]], 'row 1 has an illegal gem hand'),
                      ([good[0], good[1], tuple(bad_bit)], 'row 2 has a key bit at or above 105'),
                      ([good[0], good[1], good[2], good[1]], 'row 3 has the same key as row 1')):
        q = G.records(rows)
        with pytest.raises(S.SplendorB200Error, match=msg) as e:
            eng.solver(0, 0, 255, True, 'simple', 100, queue=q)
        assert e.value.code == -1
    run = Run(eng, capfd, good)
    try:
        run.step()
    finally:
        run.close()
