"""GPU tests (-m gpu) of the batched speedrun search (spl_sbatch_*, State.solve_many): every game of a batch equals
its own single-game search level by level and in its line, games never share visited states, and the batch keeps
its launch count per level, its link spilling and its table-full error."""
import json
from pathlib import Path

import numpy as np
import pytest

import splendor_rl_gym_b200 as S
from common import assert_digest, level_digest

pytestmark = pytest.mark.gpu

INFO_FIELDS = ('frontier', 'generated', 'unique', 'kept', 'visited', 'goal_rank', 'ended')
M64 = (1 << 64) - 1
# every (tie policy, noise) group of the golden beam runs, read from the file so that none is left out
GOLDEN_GROUPS = sorted({(r['policy'], r['noise'])
                        for r in json.loads((Path(__file__).parent / 'golden' / 'beam_runs.json').read_text())})


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def _row(state):
    k, a = state.record()
    return (k & M64, k >> 64, a, M64)


def _rows(states):
    return np.array([_row(s) for s in states], dtype=np.uint64)


def _path_state(p):
    return S.State(cards=tuple(p['cards']), bonus=tuple(p['bonus']), gems=tuple(p['gems']), pts=p['pts'], saved=p['saved'])


def _fields(s):
    return (repr(s), s.cards, s.bonus, s.gems, s.pts, s.saved)


# (root, goal, use_heuristic, heuristic, beam): goals, heuristics and beams mixed, 1 and a beam above any level
# included, mid-game roots taken along a golden line, a BFS game with a small goal, and games that end at different
# levels
def _mixed_games(golden):
    line = next(r for r in golden['beam_runs'] if r['base'] == 'aggressive' and r['beam'] == 20000 and r['policy'] == 'stable')['path']
    mid, late = _path_state(line[6]), _path_state(line[14])
    new = S.State.newgame()
    return [(new, 6, True, 'simple', 1000), (mid, 10, True, 'balanced', 1), (new, 3, False, 'simple', 1),
            (late, 15, True, 'aggressive', 5000), (new, 4, True, 'efficiency', 10 ** 9), (mid, 12, True, 'competitive', 300),
            (new, 15, True, 'simple', 7), (late, 13, True, 'nonexistent', 2000)]


def _trace_batch(eng, games, tie, noise):
    """per game: [(counters, queue rows)] for every level it took part in, and its line rows"""
    roots, goals, kinds, names, beams = zip(*games)
    sol = eng.sbatch_solver(_rows(roots), goals, kinds, names, beams, tie, noise)
    out = [[] for _ in games]
    while not sol.ended:
        info = sol.step()
        for g, gi in enumerate(info['games']):
            if out[g] and out[g][-1][0]['ended']:
                assert {k: gi[k] for k in INFO_FIELDS} == out[g][-1][0] and len(sol.frontier(g)) == 0, g  # frozen once ended
                continue
            out[g].append(({k: gi[k] for k in INFO_FIELDS}, sol.frontier(g).tobytes()))
    lines = sol.lines()
    sol.close()
    return out, lines


def _trace_single(eng, root, goal, use_h, name, beam, tie, noise):
    k, a = root.record()
    sol = eng.solver(k, a, goal, use_h, name, beam, tie, noise)
    out = []
    while not sol.ended:
        gi = sol.step()
        fr = b'' if gi['ended'] else sol.frontier().cpu().numpy().view(np.uint64).tobytes()
        out.append(({k: gi[k] for k in INFO_FIELDS}, fr))
    sol.close()
    return out


def test_golden_groups_cover_every_run(golden):
    assert len(GOLDEN_GROUPS) == 4
    assert sum(1 for r in golden['beam_runs'] if (r['policy'], r['noise']) in GOLDEN_GROUPS) == len(golden['beam_runs']) == 37


@pytest.mark.parametrize('tie,noise', GOLDEN_GROUPS)
def test_golden_runs_as_batches(eng, golden, tie, noise):
    """The golden beam runs of one (tie, noise) group as one batch: every level of every game against the reference's
    counters and queue digests, then moves, expanded, generated, visited and the line."""
    runs = [r for r in golden['beam_runs'] if (r['policy'], r['noise']) == (tie, noise)]
    n = len(runs)
    sol = eng.sbatch_solver(_rows([S.State.newgame()] * n), [r['goal'] for r in runs], [True] * n, [r['base'] for r in runs],
                            [r['beam'] for r in runs], tie, noise)
    expanded, generated, done = [0] * n, [0] * n, [None] * n
    level = 0
    while not sol.ended:
        info = sol.step()
        for g, run in enumerate(runs):
            gi = info['games'][g]
            if done[g] is not None:
                assert gi == done[g], g
                continue
            want = run['levels'][level]
            what = f"{run['base']}@{tie}/{noise} goal={run['goal']} beam={run['beam']} level {level}"
            assert (gi['frontier'], gi['generated'], gi['unique']) == (want['frontier'], want['generated'], want.get('unique', {'n': 0})['n']), what
            assert gi['goal_rank'] == (-1 if want['goal_rank'] is None else want['goal_rank']), what
            expanded[g] += gi['frontier'] if gi['goal_rank'] < 0 else 0
            generated[g] += gi['generated']
            assert expanded[g] == sum(lv['expanded'] for lv in run['levels'][:level + 1]), what
            if gi['ended']:
                done[g] = gi
                continue
            fr = sol.frontier(g)
            assert_digest(level_digest(fr[:, 0], fr[:, 1], fr[:, 2], fr[:, 3]), want['kept'], what)
        level += 1
    lines = sol.lines()
    sol.close()
    for g, run in enumerate(runs):
        what = f"{run['base']}@{tie}/{noise} goal={run['goal']} beam={run['beam']}"
        assert done[g] is not None and done[g]['level'] == run['moves'], what
        assert (expanded[g], generated[g], done[g]['visited']) == (run['expanded'], run['generated'], run['visited']), what
        path = [S.State.from_record(int(r[0]), int(r[1]), int(r[2])) for r in lines[g]]
        assert [repr(s) for s in path] == [p['repr'] for p in run['path']], what
        assert [(s.saved, s.pts, list(s.bonus)) for s in path] == [(p['saved'], p['pts'], p['bonus']) for p in run['path']], what


@pytest.mark.parametrize('tie,noise', GOLDEN_GROUPS)
def test_levels_equal_single_solver(eng, golden, tie, noise):
    """A mixed batch against Engine.solver() stepped alone for each game: at every level the game's queue rows (key,
    aux, in-game link) byte for byte, its counters and its goal rank."""
    games = _mixed_games(golden)
    got, lines = _trace_batch(eng, games, tie, noise)
    ends = set()
    for g, (root, goal, use_h, name, beam) in enumerate(games):
        want = _trace_single(eng, root, goal, use_h, name, beam, tie, noise)
        assert len(got[g]) == len(want), g
        for lvl, ((gi, gfr), (wi, wfr)) in enumerate(zip(got[g], want)):
            assert gi == wi, (g, lvl)
            assert gfr == wfr, (g, lvl)
        assert len(lines[g]) == len(want)
        ends.add(len(want))
    assert len(ends) > 2  # the games end at different levels


def test_two_copies_are_isolated(eng, golden):
    """The same game twice in one batch, with another game between them: both copies have the counters and line of
    the game run alone (a shared visited set would let the second copy find every state already visited)."""
    games = _mixed_games(golden)
    a, b = games[0], games[3]
    got, lines = _trace_batch(eng, [a, b, a], 'stable', 'const')
    want = _trace_single(eng, *a, 'stable', 'const')
    assert got[0] == got[2] == want
    assert lines[0].tobytes() == lines[2].tobytes()


def test_two_beam_widths_of_one_root(eng):
    """One root and heuristic at two beam widths: each width gets its own result, equal to its own solve."""
    root = S.State.newgame()
    stats = []
    lines = S.State.solve_many([root, root], 10, use_heuristic=True, heuristic_name='balanced', beam_width=[50, 5000], engine=eng,
                               stats=stats)
    for g, (line, beam) in enumerate(zip(lines, (50, 5000))):
        want_stats = []
        want = root.solve(10, use_heuristic=True, heuristic_name='balanced', beam_width=beam, verbose=False, engine=eng,
                          stats=want_stats)
        assert [_fields(s) for s in line] == [_fields(s) for s in want]
        assert stats[-1]['games'][g]['visited'] == want_stats[-1]['visited']
    assert stats[-1]['games'][0]['visited'] != stats[-1]['games'][1]['visited']


def test_root_at_goal_ends_at_level_zero(eng):
    """A root that already has its goal's points ends at level 0 with the line [root]; the other game is unchanged."""
    root = S.State(cards=(), bonus=(0,) * 5, gems=(1, 0, 2, 0, 0), pts=5, saved=3)
    stats = []
    lines = S.State.solve_many([root, S.State.newgame()], [5, 6], use_heuristic=True, beam_width=1000, engine=eng, stats=stats)
    assert lines[0] == [root] and lines[0][0] is root
    g0 = stats[0]['games'][0]
    assert (g0['level'], g0['goal_rank'], g0['ended'], g0['visited']) == (0, 0, 1, 1)
    want = S.State.newgame().solve(6, use_heuristic=True, beam_width=1000, verbose=False, engine=eng)
    assert [_fields(s) for s in lines[1]] == [_fields(s) for s in want]


@pytest.mark.parametrize('kw', [dict(goal_pts=8, use_heuristic=True, heuristic_name='aggressive', beam_width=2000),
                                dict(goal_pts=3)])
def test_batch_of_one_equals_solve(eng, kw):
    stats, want_stats = [], []
    got = S.State.solve_many([S.State.newgame()], engine=eng, stats=stats, **kw)[0]
    want = S.State.newgame().solve(verbose=False, engine=eng, stats=want_stats, **kw)
    assert [_fields(s) for s in got] == [_fields(s) for s in want]
    assert [{k: d['games'][0][k] for k in INFO_FIELDS} for d in stats] == [{k: d[k] for k in INFO_FIELDS} for d in want_stats]


@pytest.mark.parametrize('tie,noise', [('stable', 'const'), ('det', 'hash')])
def test_solve_many_lines_equal_solve(eng, golden, tie, noise):
    """State.solve_many's lines for the mixed batch equal State.solve's: repr and every field of every state."""
    games = _mixed_games(golden)
    roots, goals, kinds, names, beams = (list(x) for x in zip(*games))
    lines = S.State.solve_many(roots, goals, use_heuristic=kinds, heuristic_name=names, beam_width=beams, tie_policy=tie,
                               noise=noise, engine=eng)
    for g, (root, goal, use_h, name, beam) in enumerate(games):
        want = root.solve(goal, use_heuristic=use_h, heuristic_name=name, beam_width=beam, tie_policy=tie, noise=noise,
                          verbose=False, engine=eng)
        assert lines[g][0] is root
        assert [_fields(s) for s in lines[g]] == [_fields(s) for s in want], g


def test_launches_per_level_do_not_grow_with_games():
    """A level costs the same launches for 2 games as for 32 (same root and heuristic, a table that does not grow)."""
    e = S.Engine(0, table_slots=1 << 22)
    try:
        deltas = {}
        for B in (2, 32):
            sol = e.sbatch_solver(_rows([S.State.newgame()] * B), [10] * B, [True] * B, ['balanced'] * B, [1000] * B, 'det', 'hash')
            d = []
            for _ in range(8):
                n0 = e.launch_count()
                sol.step()
                d.append(e.launch_count() - n0)
            sol.close()
            deltas[B] = d
        assert deltas[2] == deltas[32], deltas
    finally:
        e.close()


def test_link_spill_keeps_lines(golden):
    """With a 64 KB link budget the older link columns move to host memory; the lines stay the same."""
    games = _mixed_games(golden)
    roots, goals, kinds, names, beams = (list(x) for x in zip(*games))
    e = S.Engine(0)
    try:
        kw = dict(use_heuristic=kinds, heuristic_name=names, beam_width=beams, engine=e)
        want = S.State.solve_many(roots, goals, **kw)
        e.set_link_budget(64 << 10)
        got = S.State.solve_many(roots, goals, **kw)
        assert e.spilled_bytes() > 0
        for w, g in zip(want, got):
            assert [_fields(s) for s in g] == [_fields(s) for s in w]
    finally:
        e.close()


def test_table_full_leaves_engine_usable(golden):
    """Under a 2 MB table ceiling a batch of wide searches fails with SPL_E_TABLE_FULL; a small batch on the same
    Engine afterwards still returns the reference's lines."""
    runs = golden['beam_runs']
    big = [r for r in runs if r['beam'] == 20000][:3]
    small = [r for r in runs if r['visited'] < 30000]  # 2 MB hold 65 536 buckets, 39 321 states at the 0.6 load factor
    assert small
    e = S.Engine(0, max_table_bytes=2 << 20)
    try:
        with pytest.raises(S.SplendorB200Error) as ei:
            S.State.solve_many([S.State.newgame()] * len(big), [r['goal'] for r in big], use_heuristic=True,
                               heuristic_name=[r['base'] for r in big], beam_width=[r['beam'] for r in big], engine=e)
        assert ei.value.code == -5
        for run in small:
            line = S.State.solve_many([S.State.newgame()], run['goal'], use_heuristic=True, heuristic_name=run['base'],
                                      beam_width=run['beam'], tie_policy=run['policy'], noise=run['noise'], engine=e)[0]
            assert [repr(s) for s in line] == [p['repr'] for p in run['path']]
    finally:
        e.close()
