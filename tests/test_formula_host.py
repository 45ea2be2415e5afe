"""CPU tests of formula heuristics (splendor-rl-gym_b200/formula.py): validation, the plain-Python reference function
against the C oracle of formulas (tests/formula_oracle.py) bit for bit, and the four built-in twins against the
built-ins of the oracle."""
import math
import random
from types import SimpleNamespace

import numpy as np
import pytest

import formula_oracle
import oracle
from splendor_rl_gym_b200 import HEURISTICS, Formula
from splendor_rl_gym_b200.formula import BUILTIN_TWINS, FEATURES

#: formulas with negative coefficients, three-factor terms and per-colour features
MIXED = [
    Formula([(-3.5, ('pts', 2.0)), (0.25, ('saved', 0.5), ('cards', 1.1), ('colors', 0.3)), (-7, ('gem_red', 1.5))]),
    Formula([(1e-3, ('bonus_white', 2.0), ('bonus_black', 1.0)), (-2.0, ('gems', 0.9)), (4.0, ('resources', 0.45)),
             (1.5, ('gem_white', 0.0), ('bonus_green', 3.0), ('gem_blue', 0.7))]),
    Formula([(-1.0, ('saved', 1.0)), (-1.0, ('pts', 1.0)), (-1.0, ('bonus', 1.0))]),
    Formula([(1e300, ('gem_black', 0.0))]),
]


def _ref_state(rec):
    u = oracle.unpack_state(rec)
    return SimpleNamespace(cards=u['cards'], bonus=u['bonus'], gems=u['gems'], pts=u['pts'], saved=u['saved'])


@pytest.fixture(scope='module')
def bfs6():
    s = oracle.Solver(99, use_heuristic=False)
    s.run(max_levels=6)
    st, _ = s.level(6)
    assert len(st) == 166_688
    return st


def edge_states(n=3000, seed=7):
    rng = random.Random(seed)
    recs = np.zeros(n, oracle.STATE_DTYPE)
    for i in range(n):
        edge = i % 3 == 0
        cards = tuple(sorted(rng.sample(range(90), rng.choice([0, 1, 5, 30, 90]))))
        gems = [rng.randint(0, 7) for _ in range(5)]
        while sum(gems) > 10:
            j = rng.randrange(5)
            gems[j] = max(0, gems[j] - 1)
        bonus = tuple(31 if edge else rng.randint(0, 31) for _ in range(5))
        pts = 255 if edge else rng.randint(0, 255)
        saved = 65535 if edge else rng.randint(0, 65535)
        recs[i] = oracle.pack_state(cards, bonus, tuple(gems), pts, saved)[0]
    return recs


def _reference_scores(formula, states, draws, monkeypatch):
    it = iter(int(d) for d in draws)
    monkeypatch.setattr(random, 'randint', lambda a, b: next(it))
    f = formula.reference()
    return np.array([f(_ref_state(r)) for r in states])


@pytest.mark.parametrize('bad, match', [
    ([(1.0, ('nope', 1.0))], 'unknown feature'),
    ([(1.0, ('pts', -0.5))], 'negative or not finite'),
    ([(1.0, ('pts', math.inf))], 'negative or not finite'),
    ([(1.0, ('pts', math.nan))], 'negative or not finite'),
    ([(math.inf, ('pts', 1.0))], 'coefficient is not finite'),
    ([(math.nan, ('pts', 1.0))], 'coefficient is not finite'),
    ([(1.0, ('pts', 1.0))] * 9, '1 to 8 terms'),
    ([], '1 to 8 terms'),
    ([(1.0, ('pts', 1.0), ('saved', 1.0), ('cards', 1.0), ('gems', 1.0))], 'at most 3 factors'),
    ([(1.0,)], 'factors'),
    ([(1.0, ('saved', 1000.0))], 'not a finite double'),
    ([(1e300, ('pts', 100.0))], 'not a finite double'),
    ([(0.0, ('saved', 1000.0))], 'not a finite double'),  # 0 * inf is NaN
    ([(1.7e308, ('pts', 0.0)), (1.7e308, ('saved', 0.0))], 'not a finite double'),
])
def test_validation_errors(bad, match):
    with pytest.raises(ValueError, match=match):
        Formula(bad)


def test_formula_is_an_immutable_hashable_value():
    a = Formula([(2, ('pts', 1))])
    b = Formula([(2.0, ('pts', 1.0))])
    assert a == b and hash(a) == hash(b) and len({a, b}) == 1
    assert a != Formula([(2.0, ('pts', 1.5))])
    with pytest.raises(AttributeError):
        a.terms = ()
    assert set(FEATURES) >= {'pts', 'saved', 'cards', 'gems', 'bonus', 'resources', 'colors', 'gem_black', 'bonus_white'}


def test_heuristics_registry_is_unchanged():
    assert set(HEURISTICS) == {'simple', 'balanced', 'aggressive', 'efficiency', 'competitive'}
    assert not any(isinstance(v, Formula) for v in HEURISTICS.values())


@pytest.mark.parametrize('which', ['bfs6', 'edges'])
@pytest.mark.parametrize('k', range(len(MIXED) + len(BUILTIN_TWINS)))
def test_reference_function_equals_oracle(k, which, bfs6, monkeypatch):
    formula = (MIXED + list(BUILTIN_TWINS.values()))[k]
    states = bfs6 if which == 'bfs6' else edge_states()
    if which == 'bfs6' and k % 2:
        states = states[::7]  # every formula sees part of the level, the full level is covered twice
    draws = np.random.default_rng(k).integers(1, 101, len(states))
    want = formula_oracle.score(states, formula, draws=draws)
    got = _reference_scores(formula, states, draws, monkeypatch)
    assert got.view(np.uint64).tolist() == want.view(np.uint64).tolist()
    if k == 2 and which == 'edges':
        assert (want < 0).mean() > 0.9  # negative totals


@pytest.mark.parametrize('noise', ['const', 'hash'])
@pytest.mark.parametrize('name', list(BUILTIN_TWINS))
def test_twins_equal_builtins_under_oracle(name, noise, bfs6):
    states = np.concatenate([bfs6, edge_states()])
    assert formula_oracle.score(states, BUILTIN_TWINS[name], noise).view(np.uint64).tolist() == \
        oracle.score(states, name, noise).view(np.uint64).tolist()


@pytest.mark.parametrize('policy', ['stable', 'det'])
@pytest.mark.parametrize('name', list(BUILTIN_TWINS))
def test_twin_solver_equals_builtin_level_by_level(name, policy):
    kw = dict(beam_width=300, policy=policy, noise='hash')
    a = oracle.Solver(8, use_heuristic=True, heuristic_name=name, **kw)
    b = formula_oracle.Solver(8, BUILTIN_TWINS[name], **kw)
    a.run()
    b.run()
    assert a.infos == b.infos and a.nlevels == b.nlevels
    for i in range(a.nlevels):
        sa, la = a.level(i)
        sb, lb = b.level(i)
        assert (sa == sb).all() and (la == lb).all()
    assert (a.path() == b.path()).all()
