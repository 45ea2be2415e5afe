"""GPU tests (-m gpu) of the batched realistic search (spl_rbatch_*, realistic.solve_many): every game of a batch
equals its own single-game search level by level, games never share visited states, and the batch keeps its launch
count per level, its link spilling and its table-full error."""
import hashlib

import numpy as np
import pytest

import oracle
import splendor_rl_gym_b200 as S
from common import assert_digest, rlevel_digest
from splendor_rl_gym_b200.realistic import RConfig

pytestmark = pytest.mark.gpu

INFO_FIELDS = ('frontier', 'generated', 'unique', 'kept', 'visited', 'goal_rank', 'ended')


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def _cfg(run):
    cfg = RConfig(run['players'], run['goal'], run['gems_per_color'], 0)
    for t, seq in enumerate((run['market']['t1'], run['market']['t2'], run['market']['t3'])):
        cfg.deck_len[t] = len(seq)
        for i, c in enumerate(seq):
            cfg.deck[t][i] = c
    return cfg


def _ocfg(run):
    return oracle.make_rconfig(run['players'], run['goal'], run['gems_per_color'],
                               [run['market']['t1'], run['market']['t2'], run['market']['t3']])


def _path_sha(recs, players):
    return [hashlib.sha256(r['p'][:players].tobytes() + r['vis'].tobytes() + bytes([int(r['cur'])])).hexdigest()[:16]
            for r in recs]


def _root(players, goal, seed):
    gpc = {2: 4, 3: 5, 4: 7}[players]
    cfg = S.GameConfig(num_players=players, target_points=goal, gems_per_color=gpc, infinite_resources=False)
    return S.MultiPlayerState.newgame(cfg, shuffle_market=seed is not None, seed=seed)


def _golden_root(run):
    return _root(run['players'], run['goal'], run['seed'])


def _state_key(s):
    return (s.players, s.market, s.gem_pool, s.current_player, s.turn_number, s.final_round_triggered, s.final_round_player)


def _trace_batch(eng, cfgs, roots, beams):
    """per game: [(counters, sha256 of the queue)] per level it took part in, and its line"""
    sol = eng.rbatch_solver(cfgs, roots, beams)
    out = [[] for _ in cfgs]
    while not sol.ended:
        info = sol.step()
        for g, gi in enumerate(info['games']):
            if out[g] and out[g][-1][0]['ended']:
                continue
            out[g].append((gi, hashlib.sha256(sol.frontier(g).tobytes()).hexdigest()))
    lines = sol.lines()
    sol.close()
    return out, lines


def _trace_single(eng, cfg, root, beam):
    sol = eng.rsolver(cfg, root, beam)
    out = []
    while not sol.ended:
        gi = sol.step()
        fr = b'' if gi['ended'] else sol.frontier().tobytes()
        out.append(({k: gi[k] for k in INFO_FIELDS}, hashlib.sha256(fr).hexdigest()))
    sol.close()
    return out


def test_golden_runs_as_one_batch(eng, golden):
    """The 8 golden realistic runs (2-4 players, goals 6-15, four markets, beams 20-3000) as one batch: every level of
    every game against the reference's digests and counters and the oracle's visited count and queue bytes."""
    runs = golden['realistic_runs']
    roots = np.concatenate([oracle.r_root(_ocfg(r)) for r in runs])
    sol = eng.rbatch_solver([_cfg(r) for r in runs], roots, [r['beam'] for r in runs])
    orcs = [oracle.RSolver(_ocfg(r), r['beam']) for r in runs]
    last = [None] * len(runs)
    level = 0
    while not sol.ended:
        info = sol.step()
        assert info['level'] == level
        for g, run in enumerate(runs):
            gi = info['games'][g]
            what = f"game {g}: p={run['players']} goal={run['goal']} seed={run['seed']} beam={run['beam']} level {level}"
            if last[g] is not None:  # ended at an earlier level: counters frozen, no queue
                assert gi == last[g] and len(sol.frontier(g)) == 0, what
                continue
            want, oi = run['levels'][level], orcs[g].step()
            assert gi['level'] == level and gi['frontier'] == want['frontier'], what
            assert gi['goal_rank'] == (want['goal_rank'] if want['goal_rank'] is not None else -1), what
            if gi['ended']:
                assert orcs[g].done and level == run['plies'], what
                last[g] = gi
                continue
            assert (gi['generated'], gi['unique'], gi['visited']) == (want['generated'], want['unique']['n'], oi['visited']), what
            fr = sol.frontier(g)
            assert_digest(rlevel_digest(fr, run['players'], run['gems_per_color']), want['kept'], what)
            assert fr.tobytes() == orcs[g].level(oi['level'] + 1).tobytes(), what
        assert bool(info['ended']) == all(x is not None for x in last)
        level += 1
    assert all(x is not None for x in last)
    for g, (run, line) in enumerate(zip(runs, sol.lines())):
        assert len(line) - 1 == run['plies'] and _path_sha(line, run['players']) == run['path_sha'], g
    sol.close()
    for o in orcs:
        o.close()


def test_games_are_isolated(eng, golden):
    """The same root twice in one batch, plus a different game: both copies equal the single-game search (a shared
    identity would let the second copy find every state already visited)."""
    a, b = golden['realistic_runs'][4], golden['realistic_runs'][0]
    runs = [a, b, a]
    roots = np.concatenate([oracle.r_root(_ocfg(r)) for r in runs])
    got, _ = _trace_batch(eng, [_cfg(r) for r in runs], roots, [r['beam'] for r in runs])
    for g, run in enumerate(runs):
        want = _trace_single(eng, _cfg(run), oracle.r_root(_ocfg(run)), run['beam'])
        assert len(got[g]) == len(want) == run['plies'] + 1, g
        for lvl, ((gi, gs), (wi, ws)) in enumerate(zip(got[g], want)):
            assert {k: gi[k] for k in INFO_FIELDS} == wi and gs == ws, (g, lvl)


def test_batch_equals_sequential(eng):
    """24 games (2 players to 15 points and 3 players to 10, market seeds 0..11, beams 2 000 and 20 000) in one
    batch, and a batch of one, against MultiPlayerState.solve() of the same roots on the same GPU: per-level
    counters and the line."""
    games = [(p, 15 if p == 2 else 10, seed, 2000 if seed % 2 else 20_000) for p in (2, 3) for seed in range(12)]
    roots = [_root(p, goal, seed) for p, goal, seed, _ in games]
    beams = [b for *_, b in games]
    stats = []
    lines = S.solve_many(roots, beam_width=beams, engine=eng, stats=stats)
    one_stats = []
    one = S.solve_many(roots[:1], beam_width=beams[0], engine=eng, stats=one_stats)
    for g, (root, beam) in enumerate(zip(roots, beams)):
        st = []
        want = root.solve(beam_width=beam, verbose=False, engine=eng, stats=st)
        per_level = [lv['games'][g] for lv in stats[:len(st)]]
        assert [{k: d[k] for k in INFO_FIELDS} for d in per_level] == [{k: d[k] for k in INFO_FIELDS} for d in st], g
        assert [_state_key(s) for s in lines[g]] == [_state_key(s) for s in want], g
        players = root.config.num_players
        assert _path_sha([s.record()[0] for s in lines[g]], players) == _path_sha([s.record()[0] for s in want], players), g
        if g == 0:
            assert [_state_key(s) for s in one[0]] == [_state_key(s) for s in want]
            assert [d['games'][0] for d in one_stats] == per_level


def test_solve_many_api(golden):
    """solve_many returns the reference's lines, as test_multiplayer_solve_api checks for solve()."""
    params = [(2, 6, None, 300), (3, 8, 0, 400), (2, 15, 7, 20)]
    runs = [next(r for r in golden['realistic_runs'] if (r['players'], r['goal'], r['seed'], r['beam']) == p) for p in params]
    sols = S.solve_many([_golden_root(r) for r in runs], beam_width=[r['beam'] for r in runs])
    for run, sol in zip(runs, sols):
        players = run['players']
        assert len(sol) - 1 == run['plies'] and sol[-1].turn_number == run['plies']
        assert sol[-1].is_game_over() and sol[-1].get_winner() == run['winner']
        assert [dict(pts=p.pts, cards=list(p.cards), saved=p.saved, gems=list(p.gems)) for p in sol[-1].players] == run['final']
        assert _path_sha([s.record()[0] for s in sol], players) == run['path_sha']


def test_link_spill_keeps_lines(golden):
    """With a 64 KB link budget the older link columns move to host memory; the lines stay the same."""
    runs = [golden['realistic_runs'][i] for i in (1, 4, 5)]
    e = S.Engine(0)
    try:
        want = S.solve_many([_golden_root(r) for r in runs], beam_width=[r['beam'] for r in runs], engine=e)
        e.set_link_budget(64 << 10)
        got = S.solve_many([_golden_root(r) for r in runs], beam_width=[r['beam'] for r in runs], engine=e)
        assert e.spilled_bytes() > 0
        for run, w, g in zip(runs, want, got):
            assert [_state_key(s) for s in g] == [_state_key(s) for s in w]
            assert _path_sha([s.record()[0] for s in g], run['players']) == run['path_sha']
    finally:
        e.close()


def test_launches_per_level_do_not_grow_with_games(golden):
    """A level costs the same launches for 2 games as for 32 (same rules and root, a table that does not grow)."""
    run = golden['realistic_runs'][7]
    e = S.Engine(0, table_slots=1 << 22)
    try:
        deltas = {}
        for B in (2, 32):
            root = oracle.r_root(_ocfg(run))
            sol = e.rbatch_solver([_cfg(run)] * B, np.concatenate([root] * B), [run['beam']] * B)
            d = []
            for _ in range(15):
                n0 = e.launch_count()
                sol.step()
                d.append(e.launch_count() - n0)
            sol.close()
            deltas[B] = d
        assert deltas[2] == deltas[32], deltas
    finally:
        e.close()


def test_table_full_leaves_engine_usable(golden):
    """Under a 2 MB table ceiling the batch fails with SPL_E_TABLE_FULL; a single-game solve on the same Engine
    afterwards still returns the reference's line."""
    big = [golden['realistic_runs'][i] for i in (1, 4, 5)]
    e = S.Engine(0, max_table_bytes=2 << 20)
    try:
        with pytest.raises(S.SplendorB200Error) as ei:
            S.solve_many([_golden_root(r) for r in big], beam_width=[r['beam'] for r in big], engine=e)
        assert ei.value.code == -5
        run = golden['realistic_runs'][7]
        sol = _golden_root(run).solve(beam_width=run['beam'], verbose=False, engine=e)
        assert len(sol) - 1 == run['plies'] and sol[-1].get_winner() == run['winner']
        assert _path_sha([s.record()[0] for s in sol], run['players']) == run['path_sha']
    finally:
        e.close()
