"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against (a) the golden
fixtures generated from the unmodified reference and (b) the CPU oracle on the same inputs.
Integer / byte / index work is compared bit-exactly; f64 scores are compared bit-exactly too
(tolerance 0 ulp: the heuristics are reproduced in the reference's own arithmetic)."""
import numpy as np
import pytest
import torch

import oracle
import splendor_rl_gym_b200 as S
from common import assert_digest, key_str, level_digest
from splendor_rl_gym_b200.engine import _i64, pack_aux, pack_key

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def _dev(eng, recs):
    """oracle-format records -> device (keys [n,2], aux [n])"""
    keys = np.stack([recs['lo'], recs['hi']], axis=1)
    return eng.to_device(keys, recs['aux'])


def _host(t):
    return t.cpu().numpy().view(np.uint64)


# ------------------------------------------------------------------ reference golden vectors
def test_state_iter_reference_vector():
    """tests/test_solver.py:63-89 of the reference: the 23 successors of `state1`."""
    st = S.State.newgame()
    for card in (40, 5, 21):
        st = st.buy_card(card)
    st.gems = (1, 2, 0, 0, 3)
    assert {str(s) for s in st} == {
        '(2, 3, 0, 1, 3) 0W12-0B113-1W223', '(2, 2, 0, 1, 4) 0W12-0B113-1W223', '(1, 3, 1, 1, 3) 0W12-0B113-1W223',
        '(1, 2, 1, 1, 4) 0W12-0B113-1W223', '(1, 1, 0, 0, 1) 0W12-0W22-0B113-1W223',
        '(0, 2, 0, 0, 2) 0W12-0W113-0B113-1W223', '(2, 3, 1, 0, 3) 0W12-0B113-1W223',
        '(2, 2, 1, 0, 4) 0W12-0B113-1W223', '(1, 2, 0, 0, 3) 0W12-0G12-0B113-1W223', '(1, 4, 0, 0, 3) 0W12-0B113-1W223',
        '(1, 2, 0, 2, 3) 0W12-0B113-1W223', '(0, 2, 0, 0, 3) 0R3-0W12-0B113-1W223', '(3, 2, 0, 0, 3) 0W12-0B113-1W223',
        '(1, 2, 0, 0, 5) 0W12-0B113-1W223', '(1, 2, 0, 0, 0) 0B3-0W12-0B113-1W223', '(1, 0, 0, 0, 3) 0W3-0W12-0B113-1W223',
        '(2, 3, 0, 0, 4) 0W12-0B113-1W223', '(1, 0, 0, 0, 1) 0W12-0B113-1W223-1G223',
        '(1, 2, 0, 0, 1) 0W12-0B12-0B113-1W223', '(2, 2, 1, 1, 3) 0W12-0B113-1W223', '(1, 3, 1, 0, 4) 0W12-0B113-1W223',
        '(1, 2, 2, 0, 3) 0W12-0B113-1W223', '(1, 3, 0, 1, 4) 0W12-0B113-1W223'}


def test_bfs_winning_lines(golden):
    """tests/test_solver.py:92-113 of the reference: exact pure-BFS lines for goal 3 and goal 4."""
    for goal, want in golden['bfs_lines'].items():
        sol = S.State.newgame().solve(goal_pts=int(goal), verbose=False)
        assert [str(s) for s in sol] == want


def test_heuristic_properties():
    """tests/test_heuristics.py of the reference: sign, type, monotonicity, unknown-name fallback."""
    z = (0,) * 5
    for name in ('simple', 'balanced', 'aggressive', 'efficiency'):
        h = S.HEURISTICS[name]
        v = h(S.State.newgame())
        assert isinstance(v, float) and v >= 0
        lo_ = S.State(cards=(), bonus=z, gems=z, pts=2, saved=5)
        hi_ = S.State(cards=(), bonus=z, gems=z, pts=12, saved=5)
        assert h(hi_) > h(lo_)
        assert abs(h(lo_) - h(lo_)) < 1.0
    sol = S.State.newgame().solve(goal_pts=3, use_heuristic=True, heuristic_name='nonexistent', beam_width=1000, verbose=False)
    assert sol[-1].pts >= 3


# ------------------------------------------------------------------ stage operators vs golden / oracle
def test_expand_matches_reference_successors(eng, golden):
    succ = golden['successors']
    recs = np.concatenate([oracle.pack_state(s['cards'], s['bonus'], s['gems'], s['pts'], s['saved']) for s in succ])
    ck, ca, cl = (_host(t) for t in eng.expand(*_dev(eng, recs)))
    pos = 0
    for rank, s in enumerate(succ):
        for ordinal, want in enumerate(s['children']):
            assert key_str(ck[pos, 0], ck[pos, 1]) == want['key']
            aux = int(ca[pos])
            assert (aux & 0xffff, (aux >> 16) & 0xff) == (want['saved'], want['pts'])
            assert [(aux >> (24 + 5 * c)) & 31 for c in range(5)] == want['bonus']
            assert int(cl[pos]) == rank << 8 | ordinal
            pos += 1
    assert pos == len(ca)


def test_expand_edge_cases(eng):
    # empty batch, a hand of 10 gems (returns), all 7s in one colour, a hand above 10 gems, a full deck
    k, a, l = eng.expand(torch.empty((0, 2), dtype=torch.int64, device=eng.tdev), torch.empty(0, dtype=torch.int64, device=eng.tdev))
    assert k.shape[0] == 0
    cases = [((), z5(), (2, 2, 2, 2, 2), 0, 0), ((), z5(), (7, 3, 0, 0, 0), 0, 0), ((), z5(), (7, 7, 7, 7, 7), 0, 0),
             (tuple(range(90)), (18,) * 5, (0, 0, 0, 0, 0), 140, 100), ((), (7, 7, 7, 7, 7), (0, 0, 0, 0, 0), 0, 0)]
    recs = np.concatenate([oracle.pack_state(*c) for c in cases])
    ck, ca, cl = (_host(t) for t in eng.expand(*_dev(eng, recs)))
    want = [oracle.expand(recs[i:i + 1]) for i in range(len(cases))]
    assert sum(len(w) for w in want) == len(ca)
    pos = 0
    for rank, w in enumerate(want):
        for o in range(len(w)):
            assert (ck[pos, 0], ck[pos, 1], ca[pos], cl[pos]) == (w['lo'][o], w['hi'][o], w['aux'][o], rank << 8 | o)
            pos += 1
    assert len(want[2]) == 90  # total > 10: no takes, but every card is affordable
    assert len(want[3]) == 15  # owns the whole deck: only takes
    assert len(want[4]) == 90 + 15  # every card affordable on bonuses alone


def z5():
    return (0, 0, 0, 0, 0)


@pytest.mark.parametrize('noise', ['const', 'hash'])
def test_scores_bit_exact_vs_reference(eng, golden, noise):
    rows = golden['scores']
    lo = np.array([int(r['key']) & (2 ** 64 - 1) for r in rows], dtype=np.uint64)
    hi = np.array([int(r['key']) >> 64 for r in rows], dtype=np.uint64)
    aux = np.array([pack_aux(r['bonus'], r['pts'], r['saved']) for r in rows], dtype=np.uint64)
    keys, a = eng.to_device(np.stack([lo, hi], 1), aux)
    for h in ('simple', 'balanced', 'aggressive', 'efficiency'):
        got = eng.score(h, keys, a, noise).cpu().numpy().view(np.uint64)
        want = np.array([r[f'{h}:{noise}'] for r in rows], dtype=np.uint64)
        assert (got == want).all(), (h, noise, int((got != want).sum()))


def test_scores_bit_exact_vs_oracle_level6(eng):
    s = oracle.Solver(10 ** 9)
    s.run(max_levels=6)
    st, _ = s.level(6)  # 166 688 states
    keys, a = _dev(eng, st)
    for h in ('simple', 'balanced', 'aggressive', 'efficiency'):
        for noise in ('const', 'hash'):
            got = eng.score(h, keys, a, noise).cpu().numpy().view(np.uint64)
            assert (got == oracle.score(st, h, noise).view(np.uint64)).all(), (h, noise)


def test_dedup_first_arrival(eng):
    """spl_dedup == `if next_step in trail: continue; trail[...] = ...; append` in arrival order."""
    eng.reset_visited()
    rng = np.random.default_rng(7)
    s = oracle.Solver(10 ** 9)
    s.run(max_levels=5)
    st, _ = s.level(5)
    # candidate list with many duplicates; aux differs between duplicates so first arrival is visible
    idx = rng.integers(0, len(st), size=200_000)
    cand = st[idx].copy()
    cand['aux'] = np.arange(len(cand), dtype=np.uint64)
    uk, ua, us = eng.dedup(*_dev(eng, cand))
    seen, first = set(), []
    for i, j in enumerate(idx.tolist()):
        if j not in seen:
            seen.add(j)
            first.append(i)
    assert us.cpu().tolist() == first
    assert (_host(ua) == np.array(first, dtype=np.uint64)).all()
    assert (_host(uk)[:, 0] == cand['lo'][first]).all() and (_host(uk)[:, 1] == cand['hi'][first]).all()
    # second call: everything already visited, plus a ragged tail of new keys
    extra = s.level(4)[0]
    cand2 = np.concatenate([cand[:1000], extra])
    uk2, ua2, us2 = eng.dedup(*_dev(eng, cand2))
    assert us2.cpu().tolist() == list(range(1000, 1000 + len(extra)))
    assert eng.visited_count() == len(seen) + len(extra)
    # empty input
    e = eng.dedup(torch.empty((0, 2), dtype=torch.int64, device=eng.tdev), torch.empty(0, dtype=torch.int64, device=eng.tdev))
    assert e[0].shape[0] == 0
    eng.reset_visited()


@pytest.mark.parametrize('n,k', [(1, 1), (1000, 1), (1000, 999), (1000, 5000), (300_001, 100_000), (2_000_000, 300_000)])
def test_topk_stable(eng, n, k):
    """spl_topk == sorted(range(n), key=score, reverse=True)[:k] with Python's stable tie order."""
    rng = np.random.default_rng(n + k)
    # few distinct values -> massive ties (as the heuristics produce), incl. negative scores and -0.0
    vals = np.concatenate([rng.normal(size=37) * 1e3, [0.0, -0.0, 0.5, 1e-300, -1e300]])
    sc = vals[rng.integers(0, len(vals), size=n)]
    scores = torch.from_numpy(sc).to(eng.tdev)
    keys = torch.zeros((n, 2), dtype=torch.int64, device=eng.tdev)
    got = eng.topk(scores, keys, k, 'stable').cpu().numpy()
    want = np.argsort(-sc, kind='stable')[:k]
    assert (got == want).all()


@pytest.mark.parametrize('n,k', [(1000, 1), (1000, 999), (5000, 9000), (300_001, 100_000), (1_000_000, 300_000)])
def test_topk_det(eng, n, k):
    """tie policy `det`: sorted(range(n), key=lambda i: (score[i], key[i]), reverse=True)[:k]."""
    rng = np.random.default_rng(n * 7 + k)
    vals = np.concatenate([rng.normal(size=11) * 1e3, [0.0, 0.5, -2.0]])
    sc = vals[rng.integers(0, len(vals), size=n)]
    lo = rng.integers(0, 2 ** 63, size=n, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=n, dtype=np.uint64)
    hi = rng.integers(0, 2 ** 41, size=n, dtype=np.uint64)
    lo[: n // 3] = lo[0]  # equal low words: order decided by the high word, and vice versa
    hi[n // 2:] = hi[-1]
    dup = (lo == lo[0]) & (hi == hi[-1])
    lo[dup] = np.arange(dup.sum(), dtype=np.uint64)  # keys must stay unique
    keys, _ = eng.to_device(np.stack([lo, hi], 1), np.zeros(n, np.uint64))
    got = eng.topk(torch.from_numpy(sc).to(eng.tdev), keys, k, 'det').cpu().numpy()
    want = np.lexsort((lo, hi, sc))[::-1][:k]
    assert (got == want).all()


def test_topk_all_equal_and_distinct(eng):
    n = 100_000
    keys = torch.zeros((n, 2), dtype=torch.int64, device=eng.tdev)
    got = eng.topk(torch.full((n,), 0.5, dtype=torch.float64, device=eng.tdev), keys, 777, 'stable').cpu().numpy()
    assert (got == np.arange(777)).all()
    sc = np.random.default_rng(3).permutation(n).astype(np.float64)
    got = eng.topk(torch.from_numpy(sc).to(eng.tdev), keys, 5000, 'stable').cpu().numpy()
    assert (got == np.argsort(-sc, kind='stable')[:5000]).all()


# ------------------------------------------------------------------ fused solver vs golden / oracle
def _check_level(sol, orc_solver, gi, oi, want=None, what=''):
    for f in ('frontier', 'generated', 'unique', 'kept', 'goal_rank', 'visited'):
        assert gi[f] == oi[f], (what, f, gi, oi)
    if gi['ended']:
        return
    fr = sol.frontier().cpu().numpy().view(np.uint64)
    st, lk = orc_solver.level(oi['level'] + 1)
    assert (fr[:, 0] == st['lo']).all() and (fr[:, 1] == st['hi']).all(), what
    assert (fr[:, 2] == st['aux']).all(), what
    assert (fr[:, 3] == lk).all(), what
    if want is not None:
        assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want, what)


def test_bfs_levels_vs_reference_and_oracle(eng, golden):
    """Exhaustive BFS (config 2): per-level frontier, in queue order, vs the reference's digests
    (levels 0..8, 18.5 M states) and the oracle's full arrays (levels 0..7)."""
    k, a = S.State.newgame().record()
    sol = eng.solver(k, a, 10 ** 9 if False else 255, False, 'simple', 0)
    orc = oracle.Solver(255)
    for want in golden['bfs_levels']['levels']:
        gi = sol.step()
        assert (gi['frontier'], gi['generated'], gi['unique']) == (want['frontier'], want['generated'], want['unique']['n'])
        if want['level'] < 7:
            _check_level(sol, orc, gi, orc.step(), want['unique'], f"bfs level {want['level']}")
        else:
            fr = sol.frontier().cpu().numpy().view(np.uint64)
            assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want['unique'], f"bfs level {want['level']}")
    sol.close()
    orc.close()


def test_bfs_chunked_equals_unchunked(golden):
    """Chunking the frontier (epoch tags) must not change first-arrival results."""
    eng2 = S.Engine(0, table_slots=1 << 12, chunk_parents=256)  # tiny chunks + forced table growth
    k, a = S.State.newgame().record()
    sol = eng2.solver(k, a, 255, False, 'simple', 0)
    for want in golden['bfs_levels']['levels'][:7]:
        gi = sol.step()
        fr = sol.frontier().cpu().numpy().view(np.uint64)
        assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want['unique'], f"chunked bfs level {want['level']}")
    sol.close()
    eng2.close()


def _stable_runs(golden):
    return golden['beam_runs']  # both tie policies (stable = arrival order, det = key descending)


def test_beam_runs_vs_reference(eng, golden):
    """Beam search (configs 1/3/4 at CPU-feasible widths): every level's kept set in rank order,
    visited count, move count and winning line vs the unmodified reference."""
    for run in _stable_runs(golden):
        what = f"{run['base']}@{run['policy']}/{run['noise']} goal={run['goal']} beam={run['beam']}"
        k, a = S.State.newgame().record()
        sol = eng.solver(k, a, run['goal'], True, run['base'], run['beam'], run['policy'], run['noise'])
        for want in run['levels']:
            gi = sol.step()
            assert (gi['frontier'], gi['generated'], gi['unique']) == (want['frontier'], want['generated'], want['unique']['n']), what
            if not gi['ended']:
                fr = sol.frontier().cpu().numpy().view(np.uint64)
                assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want['kept'], f"{what} level {want['level']}")
        assert gi['ended'] and gi['visited'] == run['visited'], what
        sol.close()
        path = S.State.newgame().solve(goal_pts=run['goal'], use_heuristic=True, heuristic_name=run['base'],
                                       beam_width=run['beam'], verbose=False, tie_policy=run['policy'], noise=run['noise'])
        assert len(path) - 1 == run['moves'], what
        assert [repr(s) for s in path] == [p['repr'] for p in run['path']], what
        assert [(s.saved, s.pts, list(s.bonus)) for s in path] == [(p['saved'], p['pts'], p['bonus']) for p in run['path']], what


@pytest.mark.parametrize('hname,beam,policy,noise', [('aggressive', 300_000, 'stable', 'const'),
                                                     ('simple', 100_000, 'stable', 'const'),
                                                     ('balanced', 100_000, 'det', 'const'),
                                                     ('efficiency', 50_000, 'det', 'hash')])
def test_beam_vs_oracle_large(eng, hname, beam, policy, noise):
    """Config 1/3/4 at the reference's default width (beam 300 000) and both tie policies: full arrays vs the oracle."""
    k, a = S.State.newgame().record()
    sol = eng.solver(k, a, 15, True, hname, beam, policy, noise)
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name=hname, beam_width=beam, policy=policy, noise=noise)
    while True:
        gi, oi = sol.step(), orc.step()
        _check_level(sol, orc, gi, oi, None, f'{hname} beam {beam} level {gi["level"]}')
        if gi['ended']:
            assert orc.done
            break
    ranks, ords = sol.path()
    assert len(ords) == orc.nlevels - 1
    sol.close()
    orc.close()


def test_verbose_output_matches_reference_format(capsys):
    S.State.newgame().solve(goal_pts=3, verbose=True)
    out = capsys.readouterr().out
    assert 'SPEEDRUN MODE SOLVER' in out and 'Heuristic: None (pure BFS)' in out
    assert 'turn=0          (0, 0, 0, 0, 0)' in out
    assert 'max_pts=3       (0, 0, 2, 2, 0) 3K6' in out


# ------------------------------------------------------------------ multi-GPU building blocks on one GPU
@pytest.mark.parametrize('cfg', [(255, False, 'simple', 0, 'stable', 'const', 7, 1 << 20), (255, False, 'simple', 0, 'stable', 'const', 7, 3000),
                                 (15, True, 'aggressive', 20_000, 'stable', 'const', None, 1 << 20),
                                 (15, True, 'aggressive', 20_000, 'stable', 'const', None, 4096),
                                 (15, True, 'balanced', 20_000, 'det', 'hash', None, 5000),
                                 (15, True, 'aggressive', 20_000, 'stable', 'const', None, 4096, 'pyhash'),
                                 (255, False, 'simple', 0, 'stable', 'const', 6, 3000, 'pyhash')])
def test_sharded_solver_world1_vs_oracle(eng, cfg):
    """The sharded driver (routing, winner bytes, pass-wise select, global ranks) on a single rank, with the
    real CUDA backend, must reproduce the oracle level by level (2 and 3 ranks: on gloo with a CPU stand-in for the
    kernels in test_sharded_gloo.py, with the real kernels on one GPU in test_gpu_sharded_ranks.py)."""
    from splendor_rl_gym_b200.sharded import Comm, CudaBackend, ShardedSolver
    goal, use_h, hname, beam, tie, noise, max_levels, block = cfg[:8]
    identity = cfg[8] if len(cfg) > 8 else 'key'  # 'pyhash': routing + visited set on the reference's State.hash (8(f).3)
    sol = ShardedSolver(CudaBackend(eng), Comm(eng.tdev), 0, 0, goal, use_h, hname, beam, tie, noise, block_parents=block,
                        identity=identity)
    orc = oracle.Solver(goal, use_heuristic=use_h, heuristic_name=hname, beam_width=beam, policy=tie, noise=noise, identity=identity)
    while True:
        gi, oi = sol.step(), orc.step()
        fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
        for f in fields:
            assert gi[f] == oi[f], (f, gi, oi)
        if gi['ended']:
            break
        fr = sol.gather_frontier().cpu().numpy().view(np.uint64)
        st, lk = orc.level(oi['level'] + 1)
        assert (fr[:, 0] == st['lo']).all() and (fr[:, 1] == st['hi']).all() and (fr[:, 2] == st['aux']).all()
        assert (fr[:, 3] == lk).all()
        if max_levels and len(sol.infos) >= max_levels:
            break
    if gi['ended']:
        assert len(sol.path()[1]) == orc.nlevels - 1
    eng.reset_visited()


@pytest.mark.parametrize('hname,beam,rounds', [('aggressive', 20_000, 1 << 27), ('aggressive', 20_000, 3000), ('balanced', 5_000, 1 << 27),
                                               ('simple', 50_000, 20_000)])
def test_grouped_sharded_solver_world1_vs_oracle(eng, hname, beam, rounds):
    """The card-set-sharded driver (spl_gs_*: routed buy records, order-agnostic per-run dedup, merged score dictionary,
    arrival-order tie select, sample-sort ranks) on a single rank must reproduce the oracle level by level, with one and
    with many rounds per level (2 to 8 ranks on one GPU: test_gpu_sharded_ranks.py)."""
    from splendor_rl_gym_b200.sharded import Comm, GroupedShardedSolver
    sol = GroupedShardedSolver(eng, Comm(eng.tdev), 0, 0, 15, hname, beam, 'const', round_parents=rounds)
    orc = oracle.Solver(15, use_heuristic=True, heuristic_name=hname, beam_width=beam, policy='stable', noise='const')
    try:
        while True:
            gi, oi = sol.step(), orc.step()
            fields = ('frontier', 'goal_rank') if gi['ended'] else ('frontier', 'generated', 'unique', 'kept', 'goal_rank', 'visited')
            for f in fields:
                assert gi[f] == oi[f], (f, gi, oi)
            if gi['ended']:
                break
            fr = sol.gather_frontier().cpu().numpy().view(np.uint64)
            st, lk = orc.level(oi['level'] + 1)
            assert (fr[:, 0] == st['lo']).all() and (fr[:, 1] == st['hi']).all() and (fr[:, 2] == st['aux']).all()
            assert (fr[:, 3] == lk).all()
        assert len(sol.path()[1]) == orc.nlevels - 1
    finally:
        sol.close()
        orc.close()


def test_grouped_sharded_solver_reports_dictionary_overflow(eng):
    """`balanced` at beam 300 000 has more distinct scores per level than the merged score dictionary holds: the driver
    says so (State.solve() and bench.py then rerun on the key-sharded driver) and leaves the context usable."""
    from splendor_rl_gym_b200.sharded import Comm, DictionaryOverflow, GroupedShardedSolver
    sol = GroupedShardedSolver(eng, Comm(eng.tdev), 0, 0, 15, 'balanced', 300_000, 'const')
    try:
        with pytest.raises(DictionaryOverflow):
            while not sol.step()['ended']:
                pass
    finally:
        sol.close()
    k, aux = S.State.newgame().record()
    again = eng.solver(k, aux, 15, True, 'balanced', 2_000, 'stable', 'const')
    assert again.run()[-1]['ended']
    again.close()


def test_link_columns_spill_to_host_same_path(eng):
    """spl_set_link_budget (SURVEY 8(f).2): with the per-level parent links forced out to pinned host memory the winning
    line (src/solver.py:459-464) is the one found with every column on the device -- solver and sharded driver."""
    from splendor_rl_gym_b200.sharded import Comm, GroupedShardedSolver
    k, aux = S.State.newgame().record()

    def lines():
        sol = eng.solver(k, aux, 15, True, 'aggressive', 30_000, 'stable', 'const')
        sol.run()
        one = sol.path()
        sol.close()
        gs = GroupedShardedSolver(eng, Comm(eng.tdev), 0, 0, 15, 'aggressive', 30_000, 'const', round_parents=1 << 27)
        try:
            while not gs.step()['ended']:
                pass
            two = gs.path()
        finally:
            gs.close()
        return one, two

    base = lines()
    before = eng.spilled_bytes()
    eng.set_link_budget(64 << 10)
    try:
        spilled = lines()
        moved = eng.spilled_bytes() - before
    finally:
        eng.set_link_budget(0)
    assert moved > 3 * 8 * 30_000  # most levels of both solves left the device
    for a, b in zip(base, spilled):
        assert list(a[0]) == list(b[0]) and list(a[1]) == list(b[1])
    assert list(base[0][1]) == list(base[1][1])  # and both drivers walk the same line


def test_owner_partition_and_count_less(eng):
    import ctypes as C
    from splendor_rl_gym_b200.sharded import CudaBackend
    b = CudaBackend(eng)
    rng = np.random.default_rng(5)
    n = 300_000
    keys = torch.from_numpy(rng.integers(0, 2 ** 62, size=(n, 2), dtype=np.int64)).to(eng.tdev)
    keys[:, 1] &= (1 << 41) - 1
    for world in (1, 2, 3, 8):
        perm, counts = b.owner_partition(keys, world)
        assert counts.sum() == n and sorted(perm.cpu().tolist()) == list(range(n))
        # stable: within each owner segment the original order is preserved
        p = perm.cpu().numpy()
        off = 0
        for g in range(world):
            seg = p[off:off + counts[g]]
            assert (np.diff(seg) > 0).all()
            off += counts[g]
        assert counts.min() > 0.8 * n / world  # ownership is balanced
    a = torch.sort(torch.from_numpy(rng.integers(0, 1000, size=5000, dtype=np.int64)).to(eng.tdev)).values
    bb = torch.sort(torch.from_numpy(rng.integers(0, 1000, size=7000, dtype=np.int64)).to(eng.tdev)).values
    out = torch.zeros(5000, dtype=torch.int64, device=eng.tdev)
    b.count_less(1, False, (a, None, None), (bb, None, None), out, False, True)
    assert (out.cpu().numpy() == np.searchsorted(bb.cpu().numpy(), a.cpu().numpy(), side='left')).all()
    b.count_less(1, True, (a, None, None), (bb, None, None), out, True)
    want = np.searchsorted(bb.cpu().numpy(), a.cpu().numpy(), side='left') + np.searchsorted(bb.cpu().numpy(), a.cpu().numpy(), side='right')
    assert (out.cpu().numpy() == want).all()


# ------------------------------------------------------------------ edge cases of solve()
def test_solve_edge_cases(eng):
    root = S.State.newgame()
    # goal already met by the root: the loop ends at the first dequeue (src/solver.py:443-445)
    assert [repr(s) for s in root.solve(goal_pts=0, verbose=False)] == ['(0, 0, 0, 0, 0)']
    # beam of one state, both tie policies: still a legal line that reaches the goal or dies out like the oracle's
    for tie in ('stable', 'det'):
        sol = root.solve(goal_pts=3, use_heuristic=True, heuristic_name='aggressive', beam_width=1, verbose=False, tie_policy=tie)
        orc = oracle.Solver(3, use_heuristic=True, heuristic_name='aggressive', beam_width=1, policy=tie)
        orc.run()
        want = [oracle.unpack_state(r) for r in orc.path()]
        assert [(s.cards, s.gems, s.saved) for s in sol] == [(w['cards'], w['gems'], w['saved']) for w in want]
    # a hand-built root (owned cards, gems, saved) with the maximum fan-out region nearby
    st = S.State.newgame()
    for card in (40, 5, 21):
        st = st.buy_card(card)
    st.gems = (1, 2, 0, 0, 3)
    st = S.State(cards=st.cards, bonus=st.bonus, gems=st.gems, pts=st.pts, saved=st.saved)
    sol = st.solve(goal_pts=st.pts + 3, verbose=False)
    rec = oracle.pack_state(st.cards, st.bonus, st.gems, st.pts, st.saved)
    orc = oracle.Solver(st.pts + 3, root=rec)
    orc.run()
    want = [oracle.unpack_state(r) for r in orc.path()]
    assert [(s.cards, s.gems, s.saved, s.pts) for s in sol] == [(w['cards'], w['gems'], w['saved'], w['pts']) for w in want]


def test_max_fanout_state(eng):
    """190 successors (90 buys + 100 takes) -- the ordinal must fit the 8-bit link field (SURVEY.md 8a3)."""
    recs = oracle.pack_state((), (7, 7, 7, 7, 7), (2, 2, 2, 2, 2), 0, 0)
    ck, ca, cl = eng.expand(*eng.to_device(np.stack([recs['lo'], recs['hi']], 1), recs['aux']))
    want = oracle.expand(recs)
    assert len(want) == 190 == ck.shape[0]
    assert (ck.cpu().numpy().view(np.uint64)[:, 0] == want['lo']).all() and (ca.cpu().numpy().view(np.uint64) == want['aux']).all()
    assert cl.cpu().tolist() == list(range(190))


def test_table_growth_during_beam_search(golden):
    """a 64-node card-set table (beam search) must grow by rehash many times without changing any level"""
    eng2 = S.Engine(0, table_slots=4096, chunk_parents=1024, node_slots=64)
    run = next(r for r in golden['beam_runs'] if r['base'] == 'aggressive' and r['beam'] == 20000 and r['policy'] == 'stable')
    k, a = S.State.newgame().record()
    sol = eng2.solver(k, a, run['goal'], True, 'aggressive', run['beam'], 'stable', run['noise'])
    for want in run['levels']:
        gi = sol.step()
        if gi['ended']:
            break
        fr = sol.frontier().cpu().numpy().view(np.uint64)
        assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want['kept'], f"growth level {want['level']}")
    assert gi['ended'] and gi['table_slots'] > 64 * 256
    sol.close()
    eng2.close()


# ------------------------------------------------------------------ the reference's own identity (SURVEY 8f.3)
def test_pyhash_kernel_matches_reference(eng, golden):
    """spl_pyhash == hash((cards, gems)) of the reference (src/solver.py:316) on 2236 reachable states, bit for bit."""
    rows = golden['pyhash']['rows']
    keys = np.array([[int(k) & ((1 << 64) - 1), int(k) >> 64] for k, _ in rows], dtype=np.uint64)
    want = np.array([int(h) for _, h in rows], dtype=np.uint64)
    dk, _ = eng.to_device(keys, np.zeros(len(rows), np.uint64))
    assert np.array_equal(_host(eng.pyhash(dk)), want)


@pytest.mark.parametrize('use_h,beam,goal', [(True, 20_000, 12), (False, 0, 255)])
def test_solver_identity_pyhash(eng, use_h, beam, goal):
    """Visited set keyed by the reference's 64-bit hash: every level equals the oracle run with the same identity
    (which in turn equals the exact-key run: no collisions at this scale)."""
    k, a = S.State.newgame().record()
    sol = eng.solver(k, a, goal, use_h, 'aggressive', beam, 'stable', 'const', identity='pyhash')
    orc = oracle.Solver(goal, use_heuristic=use_h, heuristic_name='aggressive', beam_width=beam, identity='pyhash')
    try:
        for _ in range(7 if not use_h else 99):
            gi, oi = sol.step(), orc.step()
            _check_level(sol, orc, gi, oi, None, f'pyhash identity level {gi["level"]}')
            if gi['ended']:
                break
    finally:
        sol.close()
        orc.close()
        eng.set_identity('key')
