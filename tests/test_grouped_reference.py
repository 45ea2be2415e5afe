"""The host model of the grouped level (tests/grouped_ref.py) against itself and the CPU oracle: the GPU tests of
tests/test_gpu_grouped_runs.py build their rounds with it and compare the kernels with its reference level."""
import numpy as np
import pytest

import grouped_ref as G
import oracle

RICH_ROOT = oracle.pack_state((), (7,) * 5, (0,) * 5, 0, 0)


def test_hash_inverse_round_trips():
    rng = np.random.default_rng(1)
    for _ in range(2000):
        m0 = int(rng.integers(0, 1 << 63)) << 1 | int(rng.integers(0, 2))
        m1 = int(rng.integers(0, 1 << 26))
        h = G.hash_key(m0, m1)
        assert G.m0_for_hash(h, m1) == m0
        h2 = int(rng.integers(0, 1 << 63)) << 1 | int(rng.integers(0, 2))
        assert G.hash_key(G.m0_for_hash(h2, m1), m1) == h2
    assert G.hash_key(0, 0) == 0  # the empty card set (the new-game root's) has hash 0, sort key 0


def test_constructed_sets_have_the_intended_sort_key_and_home_slot():
    rng = np.random.default_rng(2)
    for _ in range(200):
        k = int(rng.integers(0, 1 << 30))
        h = k << G.SORT_SHIFT | int(rng.integers(0, 1 << G.SORT_SHIFT))
        m1 = int(rng.integers(0, 1 << 26))
        m0 = G.m0_for_hash(h, m1)
        lo, hi, aux, link = G.make_record(m0, m1, G.random_hand(rng), 0, 0, 200, _one_state_queue())
        assert G.card_words(lo, hi) == (m0, m1)
        assert G.set_hash(lo, hi) == h and G.sort_key(h) == k
        for nn in (64, 1 << 20, 3 * (1 << 30)):
            assert G.home_slot(h, nn) == (h * nn) >> 64 < nn
    # same top 20 bits, different sort keys: one home slot for every table of up to 2^20 slots
    hs = [(0xABCDE << 44) | (i << G.SORT_SHIFT) | i for i in range(300)]
    assert len({G.sort_key(h) for h in hs}) == 300 and len({G.home_slot(h, 1 << 20) for h in hs}) == 1


def _one_state_queue():
    q = np.zeros(1, G.REC_DTYPE)  # the new-game root: empty card set
    return q


def test_record_builder_rejects_what_the_kernels_cannot_take():
    q = _one_state_queue()
    with pytest.raises(AssertionError):
        G.make_record(5, 0, (8, 0, 0, 0, 0), 0, 0, 200, q)  # colour above 7
    with pytest.raises(AssertionError):
        G.make_record(5, 0, (3, 3, 3, 2, 0), 0, 0, 200, q)  # 11 gems
    with pytest.raises(AssertionError):
        G.make_record(5, 0, (0,) * 5, 0, 1, 200, q)          # generating state outside the queue
    with pytest.raises(AssertionError):
        G.make_record(5, 0, (0,) * 5, 0, 0, 100, q)          # a real successor's ordinal
    with pytest.raises(AssertionError):
        G.make_record(0, 0, (0,) * 5, 0, 0, 200, q)          # the generating state's own card set
    with pytest.raises(AssertionError):
        G.make_record(5, 1 << 26, (0,) * 5, 0, 0, 200, q)    # key at or above 2^105


def _queue(st, lk):
    q = np.zeros(len(st), G.REC_DTYPE)
    q['lo'], q['hi'], q['aux'], q['link'] = st['lo'], st['hi'], st['aux'], lk
    return q


@pytest.mark.parametrize('root,levels,heuristic', [(None, 5, 'simple'), (RICH_ROOT, 2, 'aggressive')])
def test_reference_level_reproduces_the_oracle(root, levels, heuristic):
    """with nothing injected and a beam above every level size, level after level equals oracle.Solver"""
    kw = dict(use_heuristic=True, heuristic_name=heuristic, beam_width=10 ** 7)
    orc = oracle.Solver(255, root=root, **kw) if root is not None else oracle.Solver(255, **kw)
    try:
        orc.run(max_levels=levels)
        st, lk = orc.level(0)
        q = _queue(st, lk)
        visited = {(int(st['lo'][0]), int(st['hi'][0]))}
        for lv in range(levels):
            q, unique = G.ref_level(q, visited, None, heuristic)
            st, lk = orc.level(lv + 1)
            info = orc.infos[lv]
            assert unique == info['unique'] and len(visited) == info['visited']
            assert np.array_equal(q, _queue(st, lk))
    finally:
        orc.close()


def test_run_prediction_counts_classes():
    """a hand-built round: one parent run, a tiny single-set run, a tiny run of two sets, a warp run and a CTA run"""
    rng = np.random.default_rng(3)
    parents = np.zeros(1, G.REC_DTYPE)  # empty card set, sort key 0
    recs = []

    def add(k, sets, n):
        ms = []
        for i in range(sets):
            m1 = i + 1
            ms.append((G.m0_for_hash(k << G.SORT_SHIFT | (i + 1), m1), m1))
        for j in range(n):
            m0, m1 = ms[j % sets]
            recs.append(G.make_record(m0, m1, G.random_hand(rng), 0, 0, 192, parents))

    add(0, 1, 3)     # joins the parent's run
    add(5, 1, 16)    # thread kernel
    add(6, 2, 4)     # tiny-sized, two sets: warp kernel
    add(7, 1, 17)    # warp kernel
    add(8, 3, 513)   # CTA kernel
    n_runs, cls, runs = G.predict_runs(parents, [20], G.records(recs))
    assert n_runs == 5 and cls == (1, 3, 1)
    assert runs[0] == (G.WARP, 2, 4, 23) and runs[5] == (G.THREAD, 1, 16, 16) and runs[6] == (G.WARP, 2, 4, 4)
    assert runs[7] == (G.WARP, 1, 17, 17) and runs[8] == (G.CTA, 3, 513, 513)
    m0, m1 = G.card_words_np(G.records(recs)['lo'], G.records(recs)['hi'])
    assert [int(h) for h in G.hash_np(m0, m1)] == [G.hash_key(a, b) for a, b in zip(m0.tolist(), m1.tolist())]


def test_queue_builder_rejects_what_the_create_rejects():
    """make_row / queue_of refuse the rows spl_solver_create_queue refuses: an illegal hand, a key bit >= 105, a key twice"""
    m = G.card_set([0, 48, 49, 89])
    with pytest.raises(AssertionError):
        G.make_row(*m, (3, 3, 3, 2, 0))          # 11 gems
    with pytest.raises(AssertionError):
        G.make_row(*m, (8, 0, 0, 0, 0))          # a colour above 7
    with pytest.raises(AssertionError):
        G.make_row(m[0], 1 << 26, (0,) * 5)      # key bit 105
    with pytest.raises(AssertionError):
        G.queue_of([G.make_row(*m, (1,) * 5), G.filler(5, 0), G.make_row(*m, (1,) * 5, (7,) * 5)])  # one key twice
    with pytest.raises(AssertionError):
        G.buyer(*G.card_set([1, 2]), 3, (0,) * 5)  # the card is not in the target set


def test_buyer_and_filler_rows():
    """a buyer of T buys its missing card into (T, hand) without paying gems; a filler has no buys and 15 takes"""
    T = G.card_set([0, 17, 48, 49, 89])
    q = G.queue_of([G.buyer(*T, c, (1, 1, 1, 0, 0)) for c in G.cards_of(*T)] + [G.filler(*G.card_set([3, 70]))])
    cands, ntk = G.expand_queue(q)
    buys = G.buys_of(q, cands)
    assert ntk[-1] == 15 and not (buys['link'] >> np.uint64(8) == np.uint64(len(q) - 1)).any()
    want = G.make_row(*T, (1, 1, 1, 0, 0))
    into_T = buys[(buys['lo'] == np.uint64(want[0])) & (buys['hi'] == np.uint64(want[1]))]
    assert [int(x) >> 8 for x in into_T['link']] == list(range(5))


def test_oracle_queue_start_reproduces_the_reference_level():
    """oracle.Solver started from a constructed queue (several rows, all visited) equals G.ref_level level by level"""
    rng = np.random.default_rng(4)
    T = G.card_set([0, 30, 48, 49, 89])
    rows = [G.buyer(*T, c, g) for c in G.cards_of(*T) for g in ((1, 1, 1, 0, 0), (0, 0, 0, 0, 0))]
    rows += [G.filler(int(rng.integers(1, 1 << 62)), int(rng.integers(0, 1 << 26))) for _ in range(20)]
    q = G.queue_of(rows)
    orc = oracle.Solver(255, use_heuristic=True, heuristic_name='aggressive', beam_width=10 ** 7, root=q)
    try:
        st, _ = orc.level(0)
        assert np.array_equal(st['lo'], q['lo']) and np.array_equal(st['aux'], q['aux'])
        visited = {(int(a), int(b)) for a, b in zip(q['lo'], q['hi'])}
        for lv in range(2):
            q, unique = G.ref_level(q, visited, None, 'aggressive')
            info = orc.step()
            assert unique == info['unique'] and len(visited) == info['visited']
            assert np.array_equal(q, _queue(*orc.level(lv + 1)))
    finally:
        orc.close()
