"""GPU tests (-m gpu): every single-game solver kind run until its queue runs out, against the CPU oracle level by level.
A search that runs out of states ends at the last state dequeued, the last row of the level it just expanded; the
golden runs all end at a goal or after a fixed number of levels, so without these tests that ending and the line walk
that starts from it would never run."""
import json
from pathlib import Path

import numpy as np
import pytest

import oracle
import splendor_rl_gym_b200 as S

pytestmark = pytest.mark.gpu

FIELDS = ('frontier', 'generated', 'unique', 'kept', 'visited', 'goal_rank')
GOLDEN = Path(__file__).parent / 'golden'
GOLDEN_GROUPS = sorted({(r['policy'], r['noise']) for r in json.loads((GOLDEN / 'beam_runs.json').read_text())})
DECK = json.loads((GOLDEN / 'tables.json').read_text())['deck']


@pytest.fixture(scope='module')
def eng():
    return S.Engine.get(0)


def rich_root(drop):
    """Every card but those in `drop` bought (bonuses and points to match), no gems: a root whose search runs out of
    states within a few dozen levels"""
    cards = tuple(c for c in range(90) if c not in drop)
    bonus = [0] * 5
    for c in cards:
        bonus[DECK[c]['bonus']] += 1
    return S.State(cards=cards, bonus=tuple(bonus), gems=(0,) * 5, pts=sum(DECK[c]['pt'] for c in cards), saved=0)


RICH_DROPS = [(0,), (0, 45, 89), (10, 20, 30, 40), (85, 86, 87, 88)]  # 89, 87, 86, 86 cards; 140, 134, 139, 120 pts


def _orc_rec(state):
    return oracle.pack_state(state.cards, state.bonus, state.gems, state.pts, state.saved)


def _run_speedrun(eng, root, goal, use_h, name, beam, tie, noise, identity='key'):
    """Engine.solver and oracle.Solver stepped together until both end: counters, queue rows (key, aux, link) and the
    line's ranks; returns the oracle so that the caller can check more"""
    k, a = root.record()
    sol = eng.solver(k, a, goal, use_h, name, beam, tie, noise, identity=identity)
    orc = oracle.Solver(goal, use_heuristic=use_h, heuristic_name=name, beam_width=beam, policy=tie, noise=noise,
                        root=_orc_rec(root), identity=identity)
    what = f'{name if use_h else "bfs"} beam={beam} {tie}/{noise} goal={goal} {identity}'
    try:
        while True:
            gi, oi = sol.step(), orc.step()
            assert {f: gi[f] for f in FIELDS} == {f: oi[f] for f in FIELDS}, (what, gi['level'])
            assert bool(gi['ended']) == orc.done, (what, gi['level'])
            if gi['ended']:
                break
            fr = sol.frontier().cpu().numpy().view(np.uint64)
            st, lk = orc.level(oi['level'] + 1)
            assert fr.tobytes() == np.stack([st['lo'], st['hi'], st['aux'], lk], 1).tobytes(), (what, gi['level'])
        assert oi['goal_rank'] == -1 and oi['kept'] == 0, what  # ran out of states
        last = len(orc.infos) - 1
        ranks, ords = sol.path()
        assert len(ords) == last and ranks[-1] == len(orc.level(last)[0]) - 1, what  # the last row dequeued
        # the line's ranks walk back through the oracle's links
        rank = ranks[-1]
        for lv in range(last, 0, -1):
            assert ranks[lv] == rank, (what, lv)
            link = int(orc.level(lv)[1][rank])
            assert ords[lv - 1] == link & 0xff, (what, lv)
            rank = link >> 8
        assert ranks[0] == rank == 0, what
    finally:
        sol.close()
        if identity != 'key':
            eng.set_identity('key')
    return orc


def _assert_line(line, orc, what):
    want = orc.path()
    last = len(orc.infos) - 1
    assert len(line) == last + 1 == len(want), what
    st, _ = orc.level(last)
    assert (want[-1]['lo'], want[-1]['hi'], want[-1]['aux']) == (st[-1]['lo'], st[-1]['hi'], st[-1]['aux']), what
    got = [(s.cards, s.bonus, s.gems, s.pts, s.saved) for s in line]
    assert got == [tuple(oracle.unpack_state(w)[f] for f in ('cards', 'bonus', 'gems', 'pts', 'saved')) for w in want], what


# ------------------------------------------------------------------ speedrun, card-set-grouped level
@pytest.mark.parametrize('tie,noise', GOLDEN_GROUPS)
def test_grouped_level_runs_out_of_states(eng, tie, noise):
    """Beam 1, 2 and 5 from the new game to goal 255: the queue runs out after 110-163 levels.  Every level against the
    oracle, then State.solve's line: it ends at the last row of the final queue and has one state per level."""
    levels = set()
    for name in ('simple', 'balanced', 'aggressive', 'efficiency'):
        for beam in (1, 2, 5):
            orc = _run_speedrun(eng, S.State.newgame(), 255, True, name, beam, tie, noise)
            levels.add(len(orc.infos))
            line = S.State.newgame().solve(255, use_heuristic=True, heuristic_name=name, beam_width=beam, verbose=False,
                                           tie_policy=tie, noise=noise, engine=eng)
            _assert_line(line, orc, f'{name} beam={beam} {tie}/{noise}')
            orc.close()
    assert min(levels) > 100


# ------------------------------------------------------------------ speedrun, key-table level
@pytest.mark.parametrize('drop', RICH_DROPS)
def test_bfs_from_card_rich_roots_runs_out(eng, drop):
    """Exhaustive BFS from a root that owns 86-89 cards: the key-table level runs out after 7-10 levels (1.7 k - 28 k
    visited states); State.solve's line ends at the last row of the final queue."""
    root = rich_root(drop)
    orc = _run_speedrun(eng, root, 255, False, 'simple', 0, 'stable', 'const')
    assert 6 <= len(orc.infos) <= 11
    _assert_line(root.solve(255, verbose=False, engine=eng), orc, f'bfs {drop}')
    orc.close()


@pytest.mark.parametrize('tie,noise', GOLDEN_GROUPS)
def test_key_table_beam_runs_out(eng, monkeypatch, tie, noise):
    """Beam search on the key-table level (SPL_NO_GROUPED=1) until the queue runs out: the new game at beams 1 and 5,
    card-rich roots at beams 3 and 1 000."""
    monkeypatch.setenv('SPL_NO_GROUPED', '1')
    for root, goal, name, beam in [(S.State.newgame(), 255, 'aggressive', 1), (S.State.newgame(), 255, 'efficiency', 5),
                                   (rich_root(RICH_DROPS[2]), 255, 'balanced', 3), (rich_root(RICH_DROPS[3]), 255, 'simple', 1000)]:
        orc = _run_speedrun(eng, root, goal, True, name, beam, tie, noise)
        line = root.solve(goal, use_heuristic=True, heuristic_name=name, beam_width=beam, verbose=False, tie_policy=tie,
                          noise=noise, engine=eng)
        _assert_line(line, orc, f'key table {name} beam={beam}')
        orc.close()


@pytest.mark.parametrize('use_h,beam', [(True, 2), (True, 1000), (False, 0)])
def test_pyhash_identity_runs_out(eng, use_h, beam):
    """The reference's own 64-bit hash as identity, until the queue runs out, against oracle.Solver(identity='pyhash')."""
    root = S.State.newgame() if beam == 2 else rich_root(RICH_DROPS[1])
    orc = _run_speedrun(eng, root, 255, use_h, 'aggressive', beam, 'stable', 'const', identity='pyhash')
    line = root.solve(255, use_heuristic=use_h, heuristic_name='aggressive', beam_width=beam, verbose=False, engine=eng,
                      identity='pyhash')
    eng.set_identity('key')
    _assert_line(line, orc, f'pyhash beam={beam}')
    orc.close()


# ------------------------------------------------------------------ realistic single game
def cut_game(players, gems, goal, seed, cut=4):
    """MultiPlayerState.newgame with its market shuffled by `seed` (None: unshuffled) and every tier's deck cut to its
    first `cut` cards, and the oracle's config of the same game"""
    st = S.MultiPlayerState.newgame(S.GameConfig(num_players=players, target_points=goal, gems_per_color=gems,
                                                 infinite_resources=False), shuffle_market=seed is not None, seed=seed)
    m = st.market
    tiers = [(m.tier1_visible + m.tier1_deck)[:cut], (m.tier2_visible + m.tier2_deck)[:cut], (m.tier3_visible + m.tier3_deck)[:cut]]
    market = S.CardMarket(*(t[:4] for t in tiers), *(t[4:] for t in tiers))
    root = S.MultiPlayerState(st.config, st.players, st.gem_pool, market, 0, 0)
    return root, oracle.make_rconfig(players, goal, gems, tiers)


@pytest.mark.parametrize('players', [2, 3, 4])
def test_realistic_runs_out_of_states(eng, players):
    """Realistic games with 1, 2 or 4 gems per colour and decks cut to their 4 visible cards, beams 1 to 50: they run
    out of states.  eng.rsolver against oracle.RSolver at every level (counters and the queue's 96-byte records), the
    line's ranks, then MultiPlayerState.solve's line against the oracle's path, record for record."""
    ends = set()
    for seed in (None, 3):
        for gems in (1, 2, 4):
            for beam in (1, 7, 50):
                root, ocfg = cut_game(players, gems, 30, seed)
                cfg = root.rconfig()
                assert bytes(cfg) == bytes(ocfg)
                sol = eng.rsolver(cfg, root.record(), beam)
                orc = oracle.RSolver(ocfg, beam)
                what = f'p={players} gems={gems} seed={seed} beam={beam}'
                try:
                    while True:
                        gi, oi = sol.step(), orc.step()
                        assert {f: gi[f] for f in FIELDS} == {f: oi[f] for f in FIELDS}, (what, gi['level'])
                        assert bool(gi['ended']) == orc.done, (what, gi['level'])
                        if gi['ended']:
                            break
                        assert sol.frontier().tobytes() == orc.level(oi['level'] + 1).tobytes(), (what, gi['level'])
                    assert oi['goal_rank'] == -1, what  # ran out of states
                    last = len(orc.infos) - 1
                    ranks, ords = sol.path()
                    assert len(ords) == last and ranks[-1] == len(orc.level(last)) - 1, what
                finally:
                    sol.close()
                want = orc.path()
                assert len(want) == last + 1 and want[-1].tobytes() == orc.level(last)[-1].tobytes(), what
                line = root.solve(beam_width=beam, verbose=False, engine=eng)
                assert [oracle.rident_bytes(s.record()[0], players) for s in line] == \
                    [oracle.rident_bytes(r, players) for r in want], what
                ends.add(last)
                orc.close()
    assert len(ends) > 1
