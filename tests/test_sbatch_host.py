"""State.solve_many (batched speedrun search): argument errors are raised on the host, before any device call, so they
need no GPU."""
import numpy as np
import pytest

import splendor_rl_gym_b200 as S

Z = (0, 0, 0, 0, 0)


def test_solve_many_is_reachable_from_the_package():
    assert 'State' in S.__all__ and callable(S.State.solve_many)
    assert S.State.solve_many.__self__ is S.State  # a classmethod


def _roots():
    return [S.State.newgame(), S.State.newgame().buy_card(40), S.State(cards=(), bonus=Z, gems=(1, 2, 0, 0, 3), pts=0, saved=0)]


@pytest.mark.parametrize('roots,kw,match', [
    ([], {}, 'at least one root'),
    (None, {'goal_pts': [6, 10]}, '2 values of goal_pts for 3 roots'),
    (None, {'use_heuristic': [True] * 4}, '4 values of use_heuristic for 3 roots'),
    (None, {'heuristic_name': ['simple', 'balanced']}, '2 values of heuristic_name for 3 roots'),
    (None, {'beam_width': [100, 200]}, '2 values of beam_width for 3 roots'),
    (None, {'beam_width': [100, 0, 100]}, '>= 1'),
    (None, {'beam_width': 0}, '>= 1'),
    (None, {'tie_policy': 'det_ordered'}, 'tie_policy'),
    (None, {'noise': 'mt'}, "'mt'"),
    (None, {'noise': 'bogus'}, 'noise'),
    ([S.State(cards=(), bonus=Z, gems=(8, 0, 0, 0, 0), pts=0, saved=0)], {}, 'root 0 has an illegal gem hand'),
    ([S.State.newgame(), S.State(cards=(), bonus=Z, gems=(3, 3, 3, 2, 0), pts=0, saved=0)], {}, 'root 1 has an illegal gem hand'),
    ([S.State(cards=(), bonus=Z, gems=(-1, 0, 0, 0, 0), pts=0, saved=0)], {}, 'illegal gem hand'),
    ([S.State(cards=(3, 90), bonus=Z, gems=Z, pts=0, saved=0)], {}, 'root 0 holds a card index outside 0..89'),
    ([S.State(cards=(-1,), bonus=Z, gems=Z, pts=0, saved=0)], {}, 'card index'),
])
def test_solve_many_argument_errors(roots, kw, match):
    if roots is None:
        roots = _roots()
    with pytest.raises(ValueError, match=match):
        S.State.solve_many(roots, **kw)


def test_too_many_roots():
    with pytest.raises(ValueError, match='at most 65536'):
        S.State.solve_many([S.State.newgame()] * ((1 << 16) + 1))


@pytest.mark.parametrize('kw', [dict(use_heuristic=np.True_), dict(goal_pts=np.int64(6)), dict(beam_width=np.int32(100)),
                                dict(heuristic_name=np.str_('balanced'))])
def test_numpy_scalars_are_one_value(kw):
    """A numpy scalar is one value for every root, as a Python scalar is: the call gets past the per-game arguments to
    the root checks, which stop it before any device call."""
    bad = S.State(cards=(), bonus=Z, gems=(8, 0, 0, 0, 0), pts=0, saved=0)
    with pytest.raises(ValueError, match='root 3 has an illegal gem hand'):
        S.State.solve_many(_roots() + [bad], **kw)
