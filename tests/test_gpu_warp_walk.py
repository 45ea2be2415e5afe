"""The warp kernel's walk (csrc/spl_m2.cuh, m2_group_warp_kernel) on level-0 queues built on purpose (-m gpu).

A step of the walk tests up to 32 candidates against the card set's bitmap with plain reads and then sets their bits
without atomics: a parent's takes by OR-ing its successor row (two rows for a paired step), buy records by OR-ing
the bits of the winners that share a bitmap word.  The queues below put into warp-class runs what that needs to get
right: paired parents whose successor rows overlap (and reach hands already in the visited set), buys whose hand a
take of an earlier or of a later parent also reaches, many buys of one step in one bitmap word (and two buys of one
state), and runs of several 32-item windows of parents and of buys.  Every level equals the CPU oracle started from
the same rows, and the round's `[grouped]` line (SPL_DEBUG) shows the run classes the host predicts, with every
constructed card set in the warp kernel's class."""
import re

import numpy as np
import pytest

import grouped_ref as G
import oracle
import splendor_rl_gym_b200 as S

pytestmark = pytest.mark.gpu

LINE = re.compile(r'\[grouped\] L(\d+) np=(\d+) items=(\d+) runs=(\d+) cls=(\d+)/(\d+)/(\d+) ')


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def _hands():
    """the legal gem hands in gemrank order (csrc/spl_tables.cuh: by hand size, then by packed key)"""
    out = []
    for total in range(11):
        for key in range(1 << 15):
            g = tuple(key >> (3 * c) & 7 for c in range(5))
            if sum(g) == total:
                out.append(g)
    return out


HANDS = _hands()
RANK = {g: i for i, g in enumerate(HANDS)}


def _take_hands(gems):
    """the hands of the gem-take successors of a row with hand `gems` (takes depend on the hand alone)"""
    q = G.queue_of([G.make_row(*G.card_set([0]), gems)])
    cands = G.expand_queue(q)[0]
    same = (cands['lo'] >> np.uint64(15) == q['lo'][0] >> np.uint64(15)) & (cands['hi'] == q['hi'][0])
    return [tuple(int(x) >> (3 * c) & 7 for c in range(5)) for x in cands['lo'][same]]


def _target(rng, n_cards):
    return G.card_set(sorted(rng.choice(90, n_cards, replace=False).tolist()))


def _buyer_rows(T, pairs):
    """buyers T \\ {card} with hand g for (card, g) in pairs: each buy is the state (T, g)"""
    return [G.buyer(*T, c, g) for c, g in pairs]


def _walk_queue(seed):
    """level-0 rows in rank order and the card sets built for the warp kernel"""
    rng = np.random.default_rng(seed)
    rows, sets = [], []
    # 1. paired steps: consecutive parents with at most 16 takes whose successor rows overlap; hand d is itself a take
    #    of a, b and c (its bit is set when the run starts: the queue is the visited set of level 0)
    P1 = _target(rng, 6)
    a, b, c, d, e, f = (1, 0, 0, 0, 0), (0, 1, 0, 0, 0), (0, 0, 1, 0, 0), (1, 1, 1, 1, 0), (0, 0, 0, 1, 0), (0, 0, 0, 0, 1)
    assert set(_take_hands(a)) & set(_take_hands(b)) and d in _take_hands(a) and d in _take_hands(c)
    assert all(len(_take_hands(g)) <= 16 for g in (a, b, c, d, e, f))
    rows += [G.make_row(*P1, g) for g in (a, b, c, d, e, f)]
    sets.append(P1)
    # 2. buys against takes: B1 arrives after p1 and reaches a take of p1 (the take wins), B2 arrives before p2 and
    #    reaches a take of p2 that p1 does not reach (the buy wins); more buyers fill the run past 16 candidates
    P2 = _target(rng, 8)
    p1, p2 = (2, 1, 0, 0, 0), (0, 0, 1, 2, 1)
    t1, t2 = _take_hands(p1), _take_hands(p2)
    h1 = t1[3]
    h2 = [h for h in t2 if h not in t1][2]
    cards = G.cards_of(*P2)
    rows += [G.make_row(*P2, p1)] + _buyer_rows(P2, [(cards[0], h1), (cards[1], h2)]) + [G.make_row(*P2, p2)]
    rows += _buyer_rows(P2, [(cards[2 + i], t2[i]) for i in range(5)])
    sets.append(P2)
    # 3. one buy step of many records in bitmap word 0 (hands of at most 3 gems: gemrank < 56) and word 1, two buyers
    #    of one state among them, between two parents whose takes reach some of those hands
    P3 = _target(rng, 12)
    cards = G.cards_of(*P3)
    small = [g for g in HANDS if sum(g) <= 3]
    word1 = [g for g in HANDS if 64 <= RANK[g] < 128][:6]
    picks = [small[i] for i in rng.choice(len(small), 20, replace=False)] + word1
    pairs = [(cards[i % len(cards)], g) for i, g in enumerate(picks)]
    pairs.append((cards[(len(picks) + 1) % len(cards)], picks[0]))  # a second buyer of (P3, picks[0]), ranked later
    assert len(set(pairs)) == len(pairs) and sum(RANK[g] < 64 for _, g in pairs) >= 16
    rows += [G.make_row(*P3, (0, 0, 0, 0, 0))] + _buyer_rows(P3, pairs) + [G.make_row(*P3, (0, 0, 1, 0, 0))]
    sets.append(P3)
    # 4. several windows: 40 parents and 120 buyers of one card set, interleaved in rank order; the buyers' hands are
    #    takes of the parents (before and after them) and repeat across buyers
    P4 = _target(rng, 30)
    cards = G.cards_of(*P4)
    par = [g for g in HANDS if sum(g) <= 4][5:45]
    pool = sorted({h for g in par[:10] for h in _take_hands(g)})
    buys = [(cards[i % len(cards)], pool[(i * 7) % len(pool)]) for i in range(120)]
    assert len(set(buys)) == len(buys)
    brows = _buyer_rows(P4, buys)
    for i, g in enumerate(par):
        rows += [G.make_row(*P4, g)] + brows[3 * i: 3 * i + 3]
    sets.append(P4)
    return rows, sets


def _front(sol):
    return np.ascontiguousarray(sol.frontier().cpu().numpy()).view(G.REC_DTYPE).reshape(-1)


@pytest.mark.parametrize('seed', [1, 2])
@pytest.mark.parametrize('hname', ['aggressive', 'simple'])
def test_warp_walk_equals_oracle(eng, capfd, monkeypatch, seed, hname):
    monkeypatch.setenv('SPL_DEBUG', '1')
    rows, sets = _walk_queue(seed)
    q = G.queue_of(rows)
    cands, ntk = G.expand_queue(q)
    n_runs, cls, runs = G.predict_runs(q, ntk, G.buys_of(q, cands), warp_max=G.WARP_MAX_ORDERED)
    for T in sets:
        k = G.sort_key(G.hash_key(*T))
        assert runs[k][:2] == (G.WARP, 1), (T, runs[k])
    assert max(runs[G.sort_key(G.hash_key(*sets[3]))][2:]) > 64
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name=hname, beam_width=10 ** 7, root=q)
    sol = eng.solver(0, 0, 15, True, hname, 10 ** 7, queue=q)
    try:
        for lv in range(2):
            gi, oi = sol.step(), orc.step()
            if lv == 0:
                lines = [tuple(int(x) for x in m.groups()) for m in LINE.finditer(capfd.readouterr().err)]
                assert len(lines) == 1 and lines[0][1:7] == (len(q), len(q) + len(G.buys_of(q, cands)), n_runs) + cls
            for f in ('frontier', 'generated', 'unique', 'kept', 'visited'):
                assert gi[f] == oi[f], (lv, f, gi, oi)
            st, lk = orc.level(lv + 1)
            fr = _front(sol)
            assert (fr['lo'] == st['lo']).all() and (fr['hi'] == st['hi']).all() and (fr['aux'] == st['aux']).all()
            assert (fr['link'] == lk).all()
    finally:
        sol.close()
        orc.close()
