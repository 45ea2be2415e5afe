"""GPU tests (-m gpu) of both batched searches (spl_sbatch_*, spl_rbatch_*) past the sizes the other tests run: a few
thousand games, and the ceiling of 65 536.  Every game is checked against its own CPU-oracle run: its counters at every
level (frozen once it has ended), its queue's rows byte for byte, and its line.  Oracle runs are cached by
configuration, so that games which share one also check that the batch keeps them apart.

What these sizes reach that small batches do not: the game pass of the segmented cut sorts over bitlen(B - 1) bits,
one 10-bit digit up to 1 024 games and two above; the line kernels run one thread per game, so more than 256 games
take more than one CTA; adjacent games with one-row queues put 32 games in one warp; long runs of ended games leave
runs of empty segments; and game ids near 65 535 go into the visited tables' hashes and stored games."""
import ctypes as C
import json
from pathlib import Path

import numpy as np
import pytest
import torch

import oracle
import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200._lib import LevelInfo, RGameInfo, check, lib
from splendor_rl_gym_b200.engine import M64, _DevArray, heuristic_id
from splendor_rl_gym_b200.realistic import RConfig

pytestmark = pytest.mark.gpu

GOLDEN = Path(__file__).parent / 'golden'
GOLDEN_GROUPS = sorted({(r['policy'], r['noise']) for r in json.loads((GOLDEN / 'beam_runs.json').read_text())})
DECK = json.loads((GOLDEN / 'tables.json').read_text())['deck']
HNAMES = ('simple', 'balanced', 'aggressive', 'efficiency', 'competitive', 'nonexistent')
COUNTERS = ('level', 'frontier', 'generated', 'unique', 'kept', 'visited', 'goal_rank', 'ended')
GAME_DTYPE = np.dtype([(f, '<i8') for f in COUNTERS[:-1]] + [('ended', '<i4'), ('pad', '<i4')])
assert GAME_DTYPE.itemsize == C.sizeof(RGameInfo)
MAX_GAMES = 1 << 16


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


# ------------------------------------------------------------------ oracle runs, cached by configuration
class Run:
    """One oracle search: `want[i]` the batch's counters of level i (COUNTERS), `queues[i]` the bytes of the queue after
    level i (while the search runs), `path` the line's rows"""

    def __init__(self, orc, row_of_level, path_rows):
        infos = orc.run()
        self.queues = [row_of_level(orc, i + 1) for i in range(len(infos) - 1)]
        want = []
        for i, oi in enumerate(infos):
            ended = int(i == len(infos) - 1)
            if oi['goal_rank'] >= 0:  # the goal is dequeued: the batch expands nothing of this game at this level
                visited = infos[i - 1]['visited'] if i else 1
                want.append((i, oi['frontier'], 0, 0, 0, visited, oi['goal_rank'], ended))
            else:
                want.append((i, oi['frontier'], oi['generated'], oi['unique'], oi['kept'], oi['visited'], -1, ended))
        self.want = np.array(want, np.int64)
        self.path = path_rows(orc.path())
        self.ran_out = infos[-1]['goal_rank'] < 0
        orc.close()

    @property
    def levels(self):
        return len(self.want)


_SRUNS, _RRUNS = {}, {}


def _srow_of_level(orc, i):
    st, lk = orc.level(i)
    return np.stack([st['lo'], st['hi'], st['aux'], lk], 1).tobytes()


def srun(root, goal, use_h, name, beam, tie, noise):
    """the oracle's speedrun search of one game (root: a State)"""
    k, a = root.record()
    key = (k, a, goal, use_h, heuristic_id(name) if use_h else -1, beam if use_h else 0, tie, noise)
    if key not in _SRUNS:
        orc = oracle.Solver(goal, use_heuristic=use_h, heuristic_name=name, beam_width=beam if use_h else 0, policy=tie,
                            noise=noise, root=oracle.pack_state(root.cards, root.bonus, root.gems, root.pts, root.saved))
        _SRUNS[key] = Run(orc, _srow_of_level, lambda p: np.stack([p['lo'], p['hi'], p['aux']], 1).tobytes())
    return _SRUNS[key]


def _rident(recs, players):
    return np.concatenate([recs['p'][:, :players].reshape(len(recs), -1).view(np.uint8).reshape(len(recs), -1),
                           recs['vis'], recs['cur'][:, None]], 1).tobytes()


def rrun(market, players, gems, goal, beam, cut):
    """the oracle's realistic search of one game; returns (Run, package RConfig, root record)"""
    key = (market, players, gems, goal, beam, cut)
    if key not in _RRUNS:
        tiers = [seq[:cut] if cut else seq for seq in MARKETS[market]]
        ocfg = oracle.make_rconfig(players, goal, gems, tiers)
        run = Run(oracle.RSolver(ocfg, beam), lambda orc, i: orc.level(i).tobytes(), lambda p: _rident(p, players))
        _RRUNS[key] = (run, RConfig.from_buffer_copy(bytes(ocfg)), oracle.r_root(ocfg))
    return _RRUNS[key]


MARKETS = [[r['market'][t] for t in ('t1', 't2', 't3')] for r in json.loads((GOLDEN / 'realistic_runs.json').read_text())]
MARKETS = [m for i, m in enumerate(MARKETS) if m not in MARKETS[:i]]  # the distinct golden markets (seeds None, 0, 3, 7)


# ------------------------------------------------------------------ stepping a batch and reading every game's queue
def _step(sol, games_fn):
    """one batch level; every game's counters as a structured array (spl_*batch_games)"""
    li = LevelInfo()
    check(lib.spl_solver_step(sol._h, C.byref(li), sol.eng._stream()), sol.eng._h)
    out = np.zeros(sol.n_games, GAME_DTYPE)
    check(games_fn(sol._h, out.ctypes.data, sol.n_games), sol.eng._h)
    sol.ended = bool(li.ended)
    return np.stack([out[f].astype(np.int64) for f in COUNTERS], 1)


def _all_queues(sol, frontier_fn, row_bytes):
    """every game's queue after the last level as bytes: one copy of the whole queue, cut where spl_*batch_frontier
    says each game's rows lie"""
    p, n = C.c_void_p(), C.c_int64()
    at = np.zeros((sol.n_games, 2), np.int64)
    for g in range(sol.n_games):
        check(frontier_fn(sol._h, g, C.byref(p), C.byref(n)), sol.eng._h)
        at[g] = (p.value or 0, n.value)
    base = at[0, 0]
    off = (at[:, 0] - base) // row_bytes
    end = int((off + at[:, 1]).max())
    if end == 0:
        return [b''] * sol.n_games
    raw = torch.as_tensor(_DevArray(int(base), (end * row_bytes,), '|u1'), device=sol.eng.tdev).cpu().numpy().tobytes()
    return [raw[o * row_bytes:(o + c) * row_bytes] for o, c in zip(off.tolist(), at[:, 1].tolist())]


def _check_batch(sol, runs, games_fn, frontier_fn, row_bytes, sample=None):
    """Step `sol` to its end: at every level every game's counters equal its run's (frozen after its last level), and
    the queue of every running game (of the games in `sample`, when given) equals its run's, byte for byte; an ended
    game's queue is empty.  Returns every game's frontier at every level (0 once it has ended)."""
    B = len(runs)
    L = max(r.levels for r in runs)
    want = np.stack([np.concatenate([r.want, np.repeat(r.want[-1:], L - r.levels, 0)]) for r in runs])  # [B, L, 8]
    levels = np.array([r.levels for r in runs])
    frontiers = []
    level = 0
    while not sol.ended:
        got = _step(sol, games_fn)
        bad = np.nonzero((got != want[:, level]).any(1))[0]
        assert len(bad) == 0, (level, bad[:8].tolist(), got[bad[:2]].tolist(), want[bad[:2], level].tolist())
        frontiers.append(np.where(got[:, 0] == level, got[:, 1], 0))  # 0: the game has ended
        if sample is None:
            queues = _all_queues(sol, frontier_fn, row_bytes)
            games = range(B)
        else:
            games = sample
        for g in games:
            q = queues[g] if sample is None else _one_queue(sol, frontier_fn, row_bytes, g)
            assert q == (runs[g].queues[level] if level < levels[g] - 1 else b''), (g, level)
        level += 1
    assert level == L
    return np.stack(frontiers)


def _one_queue(sol, frontier_fn, row_bytes, g):
    p, n = C.c_void_p(), C.c_int64()
    check(frontier_fn(sol._h, g, C.byref(p), C.byref(n)), sol.eng._h)
    if n.value == 0:
        return b''
    return torch.as_tensor(_DevArray(p.value, (n.value * row_bytes,), '|u1'), device=sol.eng.tdev).cpu().numpy().tobytes()


def _rows(states):
    rows = np.zeros((len(states), 4), np.uint64)
    for g, s in enumerate(states):
        k, a = s.record()
        rows[g] = (k & M64, k >> 64, a, M64)
    return rows


def rich_root(drop):
    """every card but those in `drop` bought, no gems: searches from it run out of states within a few dozen levels"""
    cards = tuple(c for c in range(90) if c not in drop)
    bonus = [0] * 5
    for c in cards:
        bonus[DECK[c]['bonus']] += 1
    return S.State(cards=cards, bonus=tuple(bonus), gems=(0,) * 5, pts=sum(DECK[c]['pt'] for c in cards), saved=0)


def _path_state(p):
    return S.State(cards=tuple(p['cards']), bonus=tuple(p['bonus']), gems=tuple(p['gems']), pts=p['pts'], saved=p['saved'])


# ------------------------------------------------------------------ speedrun batch of 3 000 games
def _speedrun_games(golden):
    """(root, goal, use_h, name, beam) of 3 000 games.  Runs of games already at their goal (they end at level 0) at
    the start, in the middle and at the end; 100 adjacent beam-1 games that run out of states after 100+ levels;
    goal-255 games at beams 1-5 and from card-rich roots; small goals (root pts + 1..6) at beams 1-2 000; BFS games;
    every heuristic name.  Elsewhere game g + 1 024 and g + 2 048 repeat game g."""
    line = next(r for r in golden['beam_runs'] if r['base'] == 'aggressive' and r['beam'] == 20000 and r['policy'] == 'stable')['path']
    new, mid, late = S.State.newgame(), _path_state(line[6]), _path_state(line[14])
    rich = [rich_root(d) for d in ((0,), (0, 45, 89), (10, 20, 30, 40), (85, 86, 87, 88))]
    cfgs = []
    for i, name in enumerate(HNAMES):
        cfgs += [(new, 255, True, name, b) for b in (1, 2, 5)]
        cfgs += [(r, 255, True, name, b) for r, b in zip(rich, (1, 3, 40, 1000))]
        for root in (new, mid, late):
            for k in range(1, 7):
                cfgs += [(root, root.pts + k, True, name, b) for b in (1, 3, 12, 60)]
            cfgs.append((root, root.pts + 1 + i % 3, True, name, (300, 2000)[i % 2]))
    cfgs += [(r, 255, False, 'simple', 1) for r in rich]
    cfgs += [(new, 2, False, 'simple', 1), (new, 3, False, 'simple', 1), (mid, mid.pts + 1, False, 'simple', 1)]
    at_goal = [(r, r.pts, u, HNAMES[j % 6], 1 + j) for j, (r, u) in enumerate([(new, True), (mid, False), (late, True), (rich[0], True)] * 10)]
    B = 3000
    games = [cfgs[(g % 1024 * 7) % len(cfgs)] for g in range(B)]
    games[40:140] = [(new, 255, True, HNAMES[j % 6], 1) for j in range(100)]
    for start in (0, 1480, B - 40):
        games[start:start + 40] = at_goal
    return games


@pytest.mark.parametrize('tie,noise', GOLDEN_GROUPS)
def test_speedrun_batch_of_3000_games(eng, golden, tie, noise):
    games = _speedrun_games(golden)
    B = len(games)
    runs = [srun(*gm, tie, noise) for gm in games]
    roots, goals, kinds, names, beams = (list(x) for x in zip(*games))
    # what the batch is built to hold
    assert len({h for h, u in zip(names, kinds) if u}) == 6 and not all(kinds)
    assert min(beams) == 1 and max(beams) == 2000
    assert runs[0].levels == runs[B - 1].levels == runs[1500].levels == 1
    assert sum(r.ran_out and r.levels > 100 for r in runs) >= 100
    assert sum(r.ran_out for r in runs) > 200 and sum(not r.ran_out for r in runs) > 1000
    assert any(games[g] == games[g + 1024] == games[g + 2048] and runs[g].levels > 20 for g in range(B - 2048))
    sol = eng.sbatch_solver(_rows(roots), goals, kinds, names, beams, tie, noise)
    try:
        frontiers = _check_batch(sol, runs, lib.spl_sbatch_games, lib.spl_sbatch_frontier, 32)
        # some level holds 32 adjacent games of one row each: a full warp of different games
        one = (frontiers == 1).astype(np.int64)
        runs32 = [np.convolve(one[lv], np.ones(32, np.int64), 'valid').max() for lv in range(1, len(one))]
        assert max(runs32) == 32
        lines = sol.lines()
    finally:
        sol.close()
    assert len(lines) == B
    for g, (run, line) in enumerate(zip(runs, lines)):
        assert len(line) == run.levels and np.ascontiguousarray(line[:, :3]).tobytes() == run.path, g
    got = S.State.solve_many(roots, goals, use_heuristic=kinds, heuristic_name=names, beam_width=beams, tie_policy=tie,
                             noise=noise, engine=eng)
    for g, (run, line) in enumerate(zip(runs, got)):
        assert line[0] is roots[g] and len(line) == run.levels, g
        rows = [(k & M64, k >> 64, a) for k, a in (s.record() for s in line)]
        assert np.array(rows, np.uint64).tobytes() == run.path, g


# ------------------------------------------------------------------ realistic batch of 2 000 games
def _realistic_configs():
    """the sweep of the four golden markets: 2-4 players, 1/2/4/7 gems per colour, goals 6/30/200, beams 1/3/50, full
    decks or decks cut to 4 cards; and wider beams (120, 300) on full decks"""
    out = []
    for m in range(len(MARKETS)):
        for players in (2, 3, 4):
            for gems in (1, 2, 4, 7):
                for goal in (6, 30, 200):
                    out += [(m, players, gems, goal, beam, cut) for beam in (1, 3, 50) for cut in (None, 4)]
            out += [(m, players, 7, 6, 300, None), (m, players, 4, 30, 120, None)]
    return out


def test_realistic_batch_of_2000_games(eng):
    cfgs = _realistic_configs()
    B = 2000
    games = [cfgs[g * 389 % len(cfgs)] for g in range(B)]
    made = [rrun(*gm) for gm in games]
    runs = [m[0] for m in made]
    assert sum(r.ran_out for r in runs) > B // 2 and sum(not r.ran_out for r in runs) > 50
    assert max(r.levels for r in runs) > 100 and max(gm[4] for gm in games) == 300
    sol = eng.rbatch_solver([m[1] for m in made], np.concatenate([m[2] for m in made]), [gm[4] for gm in games])
    try:
        _check_batch(sol, runs, lib.spl_rbatch_games, lib.spl_rbatch_frontier, 96)
        lines = sol.lines()
    finally:
        sol.close()
    for g, (gm, run, line) in enumerate(zip(games, runs, lines)):
        assert len(line) == run.levels and _rident(line, gm[1]) == run.path, g


# ------------------------------------------------------------------ the ceiling: 65 536 games
def _sample(B):
    rng = np.random.default_rng(65536)
    return sorted({0, 1, 1023, 1024, 32767, B - 1} | set(rng.integers(0, B, 26).tolist()))


def test_speedrun_batch_at_the_ceiling(eng):
    """65 536 games from the new game: goals 3-5, beams 1-3, the six heuristic names cycling, one (tie, noise) for the
    batch.  Every game's counters at every level and its line; the full queues of games 0, 1, 1 023, 1 024, 32 767,
    65 535 and a random sample at every level."""
    B = MAX_GAMES
    combos = [(g, b, h) for g in (3, 4, 5) for b in (1, 2, 3) for h in HNAMES]
    games = [combos[(g * 5 + g // 54) % len(combos)] for g in range(B)]
    new = S.State.newgame()
    runs = [srun(new, goal, True, name, beam, 'det', 'hash') for goal, beam, name in games]
    assert len(_SRUNS) >= 36
    goals, beams, names = ([gm[i] for gm in games] for i in range(3))
    sol = eng.sbatch_solver(_rows([new]).repeat(B, 0), goals, [True] * B, names, beams, 'det', 'hash')
    try:
        _check_batch(sol, runs, lib.spl_sbatch_games, lib.spl_sbatch_frontier, 32, _sample(B))
        lines = sol.lines()
    finally:
        sol.close()
    for g, (run, line) in enumerate(zip(runs, lines)):
        assert len(line) == run.levels and np.ascontiguousarray(line[:, :3]).tobytes() == run.path, g


def test_realistic_batch_at_the_ceiling(eng):
    """65 536 2-player games with 1 or 2 gems per colour (four markets, beams 1, 3 and 20, full and cut decks): every
    game's counters at every level and its line; the full queues of the sampled games at every level."""
    B = MAX_GAMES
    cfgs = [(m, 2, gems, 15, beam, cut) for m in range(len(MARKETS)) for gems in (1, 2) for beam in (1, 3, 20) for cut in (None, 4)]
    games = [cfgs[(g * 7 + g // 48) % len(cfgs)] for g in range(B)]
    made = {c: rrun(*c) for c in cfgs}
    runs = [made[c][0] for c in games]
    sol = eng.rbatch_solver([made[c][1] for c in games], np.concatenate([made[c][2] for c in games]), [c[4] for c in games])
    try:
        _check_batch(sol, runs, lib.spl_rbatch_games, lib.spl_rbatch_frontier, 96, _sample(B))
        lines = sol.lines()
    finally:
        sol.close()
    for g, (run, line) in enumerate(zip(runs, lines)):
        assert len(line) == run.levels and _rident(line, 2) == run.path, g


def test_one_game_past_the_ceiling_is_rejected():
    """65 537 games fail with SPL_E_INVALID in both batch creates; the Engine then still solves a small batch."""
    e = S.Engine(0)
    try:
        B = MAX_GAMES + 1
        with pytest.raises(S.SplendorB200Error) as ei:
            e.sbatch_solver(_rows([S.State.newgame()]).repeat(B, 0), [3] * B, [True] * B, ['simple'] * B, [1] * B)
        assert ei.value.code == -1 and '65536' in str(ei.value)
        run, cfg, root = rrun(0, 2, 2, 15, 3, None)
        with pytest.raises(S.SplendorB200Error) as ei:
            e.rbatch_solver([cfg] * B, root.repeat(B), [3] * B)
        assert ei.value.code == -1 and '65536' in str(ei.value)
        new = S.State.newgame()
        want = srun(new, 4, True, 'balanced', 50, 'stable', 'const')
        line = S.State.solve_many([new, new], 4, use_heuristic=True, heuristic_name='balanced', beam_width=50, engine=e)[1]
        rows = [(k & M64, k >> 64, a) for k, a in (s.record() for s in line)]
        assert np.array(rows, np.uint64).tobytes() == want.path
        sol = e.rbatch_solver([cfg] * 3, root.repeat(3), [3] * 3)
        try:
            while not sol.ended:
                sol.step()
            assert all(_rident(line, 2) == run.path for line in sol.lines())
        finally:
            sol.close()
    finally:
        e.close()


# ------------------------------------------------------------------ launches per level
def _launches(e, make, levels):
    sol = make()
    try:
        d = []
        for _ in range(levels):
            n0 = e.launch_count()
            info = sol.step()
            assert not info['ended']
            d.append(e.launch_count() - n0)
        return d
    finally:
        sol.close()


@pytest.mark.parametrize('kind', ['speedrun', 'realistic'])
def test_launches_per_level_step_past_1024_games(kind):
    """Identical games at B = 2, 1 024, 1 025 and 65 536, tiny beams, a table that does not grow: a level of 2 games
    costs what one of 1 024 costs (one digit in the game pass), and one of 1 025 what one of 65 536 costs, exactly one
    launch more (a second digit)."""
    e = S.Engine(0, table_slots=1 << 25)
    try:
        d = {}
        for B in (2, 1024, 1025, MAX_GAMES):
            if kind == 'speedrun':
                d[B] = _launches(e, lambda: e.sbatch_solver(_rows([S.State.newgame()]).repeat(B, 0), [255] * B, [True] * B,
                                                            ['balanced'] * B, [1] * B, 'det', 'hash'), 6)
            else:
                _, cfg, root = rrun(0, 2, 4, 15, 2, None)
                d[B] = _launches(e, lambda: e.rbatch_solver([cfg] * B, root.repeat(B), [2] * B), 6)
        assert d[2] == d[1024], d
        assert d[1025] == d[MAX_GAMES] == [n + 1 for n in d[1024]], d
    finally:
        e.close()
