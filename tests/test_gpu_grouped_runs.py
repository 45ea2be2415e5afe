"""Per-run dedup of the card-set-grouped level (csrc/spl_m2.cuh) on rounds built on purpose (-m gpu).

The card-set-sharded driver at world 1 receives its buy records through Comm.all_to_all_rows; the tests substitute
that call to hand the owner its records shuffled, and with records added: several card sets under one 30-bit sort
key, runs at the edges of the thread / warp / CTA classes, records that arrive between a run's parents, long probe
chains in the node table.  Every level is compared with the host reference of tests/grouped_ref.py (full queue rows,
`unique`, `visited`), and every round's `[grouped]` line (SPL_DEBUG) must show the runs and run classes the host
predicts, so each test shows that it reached the path it is about."""
import re

import numpy as np
import pytest
import torch

import grouped_ref as G
import oracle
import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200.sharded import Comm, GroupedShardedSolver

pytestmark = pytest.mark.gpu

RICH_ROOT = oracle.pack_state((), (7,) * 5, (0,) * 5, 0, 0)
NEW_ROOT = oracle.pack_state((), (0,) * 5, (0,) * 5, 0, 0)
LINE = re.compile(r'\[grouped\] L(\d+) np=(\d+) items=(\d+) runs=(\d+) cls=(\d+)/(\d+)/(\d+) .*\| nodes (\d+)/(\d+)')


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


class InjectComm(Comm):
    """World-1 Comm whose all-to-all hands the owner the round's routed records rearranged by `order(round, n)` and
    followed by `extra` (first round of the level only); what it delivered is kept per round."""

    def __init__(self, device):
        super().__init__(device)
        self.order, self.extra, self.delivered, self.calls = None, None, [], 0

    def all_to_all_rows(self, send, send_counts, recv_counts):
        recs = np.ascontiguousarray(send.cpu().numpy()).view(G.REC_DTYPE).reshape(-1)
        if self.order is not None:
            recs = recs[self.order(self.calls, len(recs))]
        if self.extra is not None and len(self.extra):
            recs = np.concatenate([recs, self.extra])
            self.extra = None
        self.calls += 1
        self.delivered.append(recs)
        return torch.from_numpy(recs.view(np.int64).reshape(-1, 4).copy()).to(send.device)


def _queue(st, lk):
    q = np.zeros(len(st), G.REC_DTYPE)
    q['lo'], q['hi'], q['aux'], q['link'] = st['lo'], st['hi'], st['aux'], lk
    return q


def _root_args(root):
    return int(root['lo'][0]) | int(root['hi'][0]) << 64, int(root['aux'][0])


def _lines(capfd):
    return [tuple(int(x) for x in m.groups()) for m in LINE.finditer(capfd.readouterr().err)]


def _gathered(sol):
    return np.ascontiguousarray(sol.gather_frontier().cpu().numpy()).view(G.REC_DTYPE).reshape(-1)


class Driven:
    """A GroupedShardedSolver (one round per level) stepped beside the host reference: step(records) injects the
    records into the level's round and checks the level; the predicted runs of the round are returned."""

    def __init__(self, eng, capfd, root, heuristic='aggressive', beam=10 ** 6):
        self.comm = InjectComm(eng.tdev)
        self.sol = GroupedShardedSolver(eng, self.comm, *_root_args(root), 255, heuristic, beam, 'const')
        self.capfd, self.heuristic, self.beam = capfd, heuristic, beam
        self.queue = _queue(root, np.array([0], np.uint64))
        self.visited = {(int(root['lo'][0]), int(root['hi'][0]))}
        self.nodes = []  # node-table slots after each level

    def step(self, recs=None):
        self.comm.extra = recs
        self.comm.delivered = []
        info = self.sol.step()
        lines = _lines(self.capfd)
        cands, ntk = G.expand_queue(self.queue)
        nxt, unique = G.ref_level(self.queue, self.visited, recs, self.heuristic, beam=self.beam, expanded=cands)
        assert (info['unique'], info['visited']) == (unique, len(self.visited))
        assert np.array_equal(_gathered(self.sol), nxt)
        assert len(self.comm.delivered) == 1 and len(lines) == 1
        n_runs, cls, runs = G.predict_runs(self.queue, ntk, self.comm.delivered[0])
        assert lines[0][3:7] == (n_runs,) + cls, (lines[0], n_runs, cls)
        self.nodes.append(lines[0][8])
        self.queue = nxt
        return runs

    def close(self):
        self.sol.close()


# ------------------------------------------------------------------ constructions
class Builder:
    """Injected records for one level: fresh sort keys, card sets under them, distinct links (q, 192..255)."""

    def __init__(self, queue, seed, avoid_q=()):
        self.q, self.rng = queue, np.random.default_rng(seed)
        m0, m1 = G.card_words_np(queue['lo'], queue['hi'])
        self.q_sets = list(zip(m0.tolist(), m1.tolist()))
        cands, _ = G.expand_queue(queue)
        c0, c1 = G.card_words_np(cands['lo'], cands['hi'])
        self.used = set((G.hash_np(np.concatenate([m0, c0]), np.concatenate([m1, c1])) >> np.uint64(G.SORT_SHIFT)).tolist())
        self.links = [(q, o) for q in range(len(queue)) if q not in set(avoid_q) for o in range(G.INJECT_ORD0, 256)]
        self.rng.shuffle(self.links)

    def fresh_key(self):
        while True:
            k = int(self.rng.integers(1, 1 << 30))
            if k not in self.used:
                self.used.add(k)
                return k

    def sets(self, k, n, twin=True):
        """n card sets under sort key k; with `twin` the first two have the same 64-bit hash (so one home slot)"""
        out = []
        for i in range(n):
            h = out[0][2] if (twin and i == 1) else k << G.SORT_SHIFT | int(self.rng.integers(0, 1 << G.SORT_SHIFT))
            m1 = int(self.rng.integers(0, 1 << 26))
            out.append((G.m0_for_hash(h, m1), m1, h))
        assert len({(a, b) for a, b, _ in out}) == n and all(G.sort_key(G.hash_key(a, b)) == k for a, b, _ in out)
        return [(a, b) for a, b, _ in out]

    def recs(self, sets, n, hands=None, order='random'):
        """n records spread over `sets`, gem hands drawn from `hands` (duplicates on purpose); order 'random' or
        'desc' (descending links: every duplicate arrives out of link order)"""
        hands = hands or [G.random_hand(self.rng) for _ in range(max(2, n // 3))]
        rows = []
        for j in range(n):
            m0, m1 = sets[j % len(sets)]
            for i, (q, o) in enumerate(self.links):
                if self.q_sets[q] != (m0, m1):
                    break
            q, o = self.links.pop(i)
            rows.append(G.make_record(m0, m1, hands[int(self.rng.integers(0, len(hands)))], int(self.q['aux'][q]), q, o, self.q))
        r = G.records(rows)
        if order == 'desc':
            return r[np.argsort(r['link'])[::-1]]
        return r[self.rng.permutation(len(r))]


def _cat(*parts):
    return np.concatenate(parts)


# ------------------------------------------------------------------ 1. shuffled records, whole searches
@pytest.mark.parametrize('hname,beam,rounds', [('aggressive', 20_000, 1 << 27), ('aggressive', 20_000, 3000),
                                               ('simple', 50_000, 1 << 27), ('simple', 50_000, 20_000)])
def test_shuffled_records_whole_search(eng, capfd, monkeypatch, hname, beam, rounds):
    """Every round's records reach the owner reversed or randomly permuted; every level equals the oracle."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    comm = InjectComm(eng.tdev)
    rng = np.random.default_rng(beam + rounds)
    comm.order = lambda call, n: np.arange(n)[::-1] if call % 2 else rng.permutation(n)
    sol = GroupedShardedSolver(eng, comm, 0, 0, 15, hname, beam, 'const', round_parents=rounds)
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name=hname, beam_width=beam, policy='stable', noise='const')
    st, lk = orc.level(0)
    queue, warp_runs = _queue(st, lk), 0
    try:
        while True:
            comm.delivered = []
            gi, oi = sol.step(), orc.step()
            lines = _lines(capfd)
            fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
            for f in fields:
                assert gi[f] == oi[f], (f, gi, oi)
            if gi['ended']:
                break
            _, ntk = G.expand_queue(queue)
            assert len(lines) == len(comm.delivered) == -(-len(queue) // rounds)
            for r, (line, recs) in enumerate(zip(lines, comm.delivered)):
                lo, hi = r * rounds, min((r + 1) * rounds, len(queue))
                n_runs, cls, _ = G.predict_runs(queue[lo:hi], ntk[lo:hi], recs)
                assert line[3:7] == (n_runs,) + cls, (gi['level'], r, line, n_runs, cls)
                warp_runs += cls[1]
            st, lk = orc.level(oi['level'] + 1)
            queue = _queue(st, lk)
            assert np.array_equal(_gathered(sol), queue)
        assert warp_runs > 100  # the warp kernel put many shuffled runs back into arrival order
    finally:
        sol.close()
        orc.close()


# ------------------------------------------------------------------ 2. several card sets under one sort key
def _shared_key_plan(b):
    """(records, {sort key: (class, sets)}) of level 1 from the rich root: 2..5 sets under one key in a tiny-sized
    run, a warp run and a CTA run; 17 sets in a CTA run; records of 1..3 other sets in the run of the empty set
    (the 15 parents whose cards are the root's), generated by those parents"""
    parts, want, plan = [], {}, []
    for n in (2, 3, 4, 5):
        for cls, count in ((G.WARP, 3 * n), (G.WARP, 60 + n), (G.CTA, 520 + 7 * n)):
            k = b.fresh_key()
            s = b.sets(k, n)
            parts.append(b.recs(s, count))
            want[k] = (cls, n)
            plan.append((s, count))
    k = b.fresh_key()
    s = b.sets(k, 17)
    parts.append(b.recs(s, 17 * 40))
    want[k], plan = (G.CTA, 17), plan + [(s, 17 * 40)]
    empty = [q for q, m in enumerate(b.q_sets) if m == (0, 0)]
    assert len(empty) == 15
    others = [(G.m0_for_hash(int(b.rng.integers(0, 1 << G.SORT_SHIFT)), m1), m1) for m1 in (1, 2, 3)]
    b.links = [(q, o) for q, o in b.links if q in empty] + [(q, o) for q, o in b.links if q not in empty]
    parts.append(b.recs(others, 30))   # generated by parents of the run they land in
    plan.append((others, 30))
    want[0] = (G.WARP, 4)
    return _cat(*parts), want, plan


def test_shared_sort_keys(eng, capfd, monkeypatch):
    """Runs holding 2..5 card sets (the warp kernel's limit), and 17 (the CTA kernel's), in every run class, two of
    them with the same 64-bit hash; a parent run holding other sets.  At the next level the same card sets and gem
    hands come again with new links: nothing may win a second time."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    d = Driven(eng, capfd, RICH_ROOT)
    try:
        d.step()
        b = Builder(d.queue, 11)
        recs, want, plan = _shared_key_plan(b)
        runs = d.step(recs)
        for k, (cls, n) in want.items():
            assert runs[k][:2] == (cls, n), (k, runs[k], cls, n)
        # the same sets and hands again, generated by states of the new queue that are not injected winners
        keyset = {(int(r['lo']), int(r['hi'])) for r in recs}
        b2 = Builder(d.queue, 12, avoid_q=[q for q in range(len(d.queue)) if (int(d.queue['lo'][q]), int(d.queue['hi'][q])) in keyset])
        again = recs.copy()
        for i in range(len(again)):
            m0, m1 = G.card_words(again['lo'][i], again['hi'][i])
            for j, (q, o) in enumerate(b2.links):
                if b2.q_sets[q] != (m0, m1):
                    break
            q, o = b2.links.pop(j)
            again['link'][i] = q << 8 | o
        before = d.sol.infos[-1]['visited']
        d.step(again[b2.rng.permutation(len(again))])
        won = {(int(r['lo']), int(r['hi'])) for r in _gathered(d.sol) if int(r['link']) & 0xff >= G.INJECT_ORD0}
        assert not won and d.sol.infos[-1]['visited'] > before
    finally:
        d.close()


# ------------------------------------------------------------------ 3. limits
@pytest.mark.parametrize('n_sets,count,cls', [(6, 6 * 5, G.WARP), (18, 18 * 35, G.CTA)])
def test_too_many_sets_under_one_sort_key(eng, capfd, monkeypatch, n_sets, count, cls):
    """One more card set under a sort key than the kernel of its class walks: the round fails and says so; the
    Engine then runs a normal search that matches the oracle."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    d = Driven(eng, capfd, RICH_ROOT)
    try:
        d.step()
        b = Builder(d.queue, 21)
        k = b.fresh_key()
        recs = b.recs(b.sets(k, n_sets), count)
        d.comm.extra = recs
        with pytest.raises(S.SplendorB200Error, match='more than 5 card sets share one 30-bit sort key .* more than 17 '):
            d.sol.step()
        _, ntk = G.expand_queue(d.queue)
        lines = _lines(capfd)
        n_runs, counts, runs = G.predict_runs(d.queue, ntk, d.comm.delivered[-1])
        assert len(lines) == 1 and lines[0][3:7] == (n_runs,) + counts and runs[k][:2] == (cls, n_sets)
    finally:
        d.close()
    monkeypatch.delenv('SPL_DEBUG')
    sol = GroupedShardedSolver(eng, Comm(eng.tdev), 0, 0, 15, 'aggressive', 20_000, 'const')
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name='aggressive', beam_width=20_000, policy='stable', noise='const')
    try:
        while True:
            gi, oi = sol.step(), orc.step()
            assert (gi['frontier'], gi['goal_rank']) == (oi['frontier'], oi['goal_rank'])
            if gi['ended']:
                break
            assert (gi['unique'], gi['visited']) == (oi['unique'], oi['visited'])
            st, lk = orc.level(oi['level'] + 1)
            assert np.array_equal(_gathered(sol), _queue(st, lk))
    finally:
        sol.close()
        orc.close()


# ------------------------------------------------------------------ 4. class edges
def test_buy_only_class_edges(eng, capfd, monkeypatch):
    """Buy-only runs of one card set with 16 / 17 records (thread / warp kernel) and 512 / 513 (warp / CTA kernel when
    records arrive unordered), duplicate hands arriving in descending link order, so the first arrival of every
    duplicated hand is the LAST of its copies to reach the owner (and copies straddle the 32-lane windows)."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    d = Driven(eng, capfd, RICH_ROOT)
    try:
        d.step()
        b = Builder(d.queue, 31)
        parts, want = [], {}
        for n, cls in ((16, G.THREAD), (17, G.WARP), (512, G.WARP), (513, G.CTA), (16, G.THREAD), (40, G.WARP)):
            k = b.fresh_key()
            hands = [G.random_hand(b.rng) for _ in range(max(3, n // 8))]
            parts.append(b.recs(b.sets(k, 1), n, hands, order='desc'))
            want[k] = (cls, 1, n, n)
        runs = d.step(_cat(*parts))
        for k, w in want.items():
            assert runs[k] == w, (k, runs[k], w)
    finally:
        d.close()


def _parent_pairs(queue, ntk):
    """(P0, P1, Q): consecutive parents of one card set, both with at most 16 takes, and a state Q of another card
    set ranked between them"""
    m0, m1 = G.card_words_np(queue['lo'], queue['hi'])
    by_set = {}
    for r, s in enumerate(zip(m0.tolist(), m1.tolist())):
        by_set.setdefault(s, []).append(r)
    for s, ranks in by_set.items():
        for p0, p1 in zip(ranks, ranks[1:]):
            if ntk[p0] <= 16 and ntk[p1] <= 16 and p1 - p0 > 1:
                return s, p0, p1, p0 + 1
    raise AssertionError('no parent pair of one card set with a state of another set between them')


@pytest.mark.parametrize('between', [True, False])
def test_parent_run_with_records(eng, capfd, monkeypatch, between):
    """A parent run (the empty card set) whose records arrive before, between and after its parents and share their
    take hands; and a record between two parents of at most 16 takes each (the warp kernel's paired step), or the
    same run without it."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    d = Driven(eng, capfd, NEW_ROOT)
    try:
        for _ in range(3):
            d.step()  # level 3: 790 states of 41 card sets
        cands, ntk = G.expand_queue(d.queue)
        s, p0, p1, q = _parent_pairs(d.queue, ntk)
        def take_hands(p, cards):
            return [tuple(int(c['lo']) >> (3 * i) & 7 for i in range(5)) for c in cands[cands['link'] >> np.uint64(8) == p]
                    if G.card_words(c['lo'], c['hi']) == cards]

        rows = []
        if between:  # shares a hand with a take of p1: it arrives first, so the record wins that hand
            rows.append(G.make_record(*s, take_hands(p1, s)[0], int(d.queue['aux'][q]), q, 200, d.queue))
        # the pair's run: records from states ranked before p0 and after p1 with the pair's take hands
        m0, m1 = G.card_words_np(d.queue['lo'], d.queue['hi'])
        outside = [r for r in range(len(d.queue)) if (int(m0[r]), int(m1[r])) != s and (r < p0 or r > p1)]
        pair_hands = take_hands(p0, s) + take_hands(p1, s)
        for j, qq in enumerate(outside[:2] + outside[-2:]):
            rows.append(G.make_record(*s, pair_hands[j % len(pair_hands)], int(d.queue['aux'][qq]), qq, 220, d.queue))
        # the empty set's parents: records from states of other sets ranked before, among and after them
        empty = [r for r in range(len(d.queue)) if G.card_words(d.queue['lo'][r], d.queue['hi'][r]) == (0, 0)]
        others = [r for r in range(len(d.queue)) if r not in set(empty)]
        hands = take_hands(empty[0], (0, 0)) + take_hands(empty[-1], (0, 0))
        picks = [others[0], others[-1]] + [r for r in others if empty[0] < r < empty[-1]][:6]
        for j, qq in enumerate(picks):
            for o in range(3):
                rows.append(G.make_record(0, 0, hands[(3 * j + o) % len(hands)], int(d.queue['aux'][qq]), qq, 210 + o, d.queue))
        recs = G.records(rows)
        runs = d.step(recs[np.random.default_rng(5).permutation(len(recs))])
        assert runs[0][0] in (G.WARP, G.CTA) and runs[0][1] == 1
        k = G.sort_key(G.hash_key(*s))
        assert runs[k][0] == G.WARP
    finally:
        d.close()


# ------------------------------------------------------------------ 5. probe chains
def test_probe_chains_across_rehashes(capfd, monkeypatch):
    """A few hundred card sets with the same top 20 hash bits and different sort keys: different runs claim nodes
    concurrently along one probe sequence of a 64-slot table that grows by rehash; their visited bits must survive
    into the next levels."""
    monkeypatch.setenv('SPL_DEBUG', '1')
    eng2 = S.Engine(0, node_slots=64)
    d = Driven(eng2, capfd, NEW_ROOT)
    try:
        d.step()
        d.step()
        b = Builder(d.queue, 41)
        top = int(b.rng.integers(1, 1 << 20)) << 44
        sets = []
        for i in range(300):
            h = top | (i + 1) << G.SORT_SHIFT | int(b.rng.integers(0, 1 << G.SORT_SHIFT))
            m1 = int(b.rng.integers(0, 1 << 26))
            sets.append((G.m0_for_hash(h, m1), m1))
        hands = [G.random_hand(b.rng) for _ in range(4)]
        first = _cat(*[b.recs([s], 2, hands) for s in sets])
        runs = d.step(first)
        assert sum(1 for s in sets if runs[G.sort_key(G.hash_key(*s))][:2] == (G.THREAD, 1)) == 300
        for lv in range(2):  # the same records with new links, plus new hands of the same sets
            keys = {(int(r['lo']), int(r['hi'])) for r in first}
            b = Builder(d.queue, 42 + lv, avoid_q=[q for q in range(len(d.queue)) if (int(d.queue['lo'][q]), int(d.queue['hi'][q])) in keys])
            fresh = [h for h in (G.random_hand(b.rng) for _ in range(40)) if h not in hands][:2]
            again = _cat(*[b.recs([s], 3, hands[:2] + fresh[lv:lv + 1]) for s in sets])
            d.step(again)
        assert d.nodes[-1] > d.nodes[2] > 64  # the table grew between the levels
    finally:
        d.close()
        eng2.close()


# ------------------------------------------------------------------ 6. ordered path (single-GPU driver)
def test_ordered_path_rich_root_shared_keys(eng):
    """The single-GPU solver (records in arrival order) from a root that can afford every card: nothing is cut before
    level 3 has been expanded, and level 3 holds card sets that share a sort key, as parent runs and as the buy-only
    runs of their successors; every level equals the oracle."""
    orc = oracle.Solver(255, use_heuristic=True, heuristic_name='simple', beam_width=200_000, root=RICH_ROOT)
    sol = eng.solver(*_root_args(RICH_ROOT), 255, True, 'simple', 200_000, 'stable', 'const')
    try:
        sizes = []
        for lv in range(4):
            gi, oi = sol.step(), orc.step()
            for f in ('frontier', 'generated', 'unique', 'kept', 'visited'):
                assert gi[f] == oi[f], (lv, f, gi, oi)
            st, lk = orc.level(lv + 1)
            fr = sol.frontier().cpu().numpy().view(np.uint64)
            assert (fr[:, 0] == st['lo']).all() and (fr[:, 1] == st['hi']).all() and (fr[:, 2] == st['aux']).all()
            assert (fr[:, 3] == lk).all()
            sizes.append(gi['unique'])
            if lv == 2:
                m0, m1 = G.card_words_np(st['lo'], st['hi'])
                sets = np.unique(np.stack([m0, m1], 1), axis=0)
                k = G.hash_np(sets[:, 0], sets[:, 1]) >> np.uint64(G.SORT_SHIFT)
                shared = int((np.unique(k, return_counts=True)[1] > 1).sum())
                assert (len(sets), shared) == (121_576, 12)
        assert sizes[:3] == [105, 5465, 187_950]
    finally:
        sol.close()
        orc.close()
