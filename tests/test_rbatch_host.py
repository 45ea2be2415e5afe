"""solve_many (batched realistic search): argument errors are raised on the host, before any device call, so they
need no GPU; and the per-game counter record keeps the C layout of spl_rgame_info."""
import ctypes as C

import pytest

import splendor_rl_gym_b200 as S
from splendor_rl_gym_b200._lib import RGameInfo


def _game(**kw):
    return S.MultiPlayerState.newgame(S.GameConfig(infinite_resources=False, **kw))


def test_solve_many_is_exported():
    assert 'solve_many' in S.__all__ and S.solve_many is S.realistic.solve_many


@pytest.mark.parametrize('roots,kw,match', [
    ([], {}, 'at least one game'),
    ([S.MultiPlayerState.newgame(S.GameConfig())], {}, 'infinite_resources'),
    (None, {'noise': 'mt'}, "'mt'"),
    (None, {'beam_width': [100, 200]}, '2 beam widths for 3 games'),
    (None, {'beam_width': [100, 0, 100]}, '>= 1'),
    (None, {'beam_width': 0}, '>= 1'),
])
def test_solve_many_argument_errors(roots, kw, match):
    if roots is None:
        roots = [_game(), _game(num_players=3, gems_per_color=5), _game(target_points=10)]
    with pytest.raises(ValueError, match=match):
        S.solve_many(roots, **kw)


def test_too_many_roots():
    """The 65 536-game ceiling is checked before any config or record is packed."""
    with pytest.raises(ValueError, match='at most 65536'):
        S.solve_many([_game()] * ((1 << 16) + 1))


def test_rgame_info_layout():
    """int64 level, frontier, generated, unique, kept, visited, goal_rank; int32 ended, pad"""
    assert C.sizeof(RGameInfo) == 64 and RGameInfo.ended.offset == 56
    assert set(RGameInfo().as_dict()) == {'level', 'frontier', 'generated', 'unique', 'kept', 'visited', 'goal_rank', 'ended'}
