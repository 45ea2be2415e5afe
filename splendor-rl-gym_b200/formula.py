"""Formula heuristics: user-declared sums of power terms that every speedrun search scores on the GPU.

A `Formula` is the shape the four built-in heuristics share (src/solver.py:210-286):

    t_i   = coef_i * x_i1 ** e_i1 * x_i2 ** e_i2 ...     # Python precedence: ((coef * p1) * p2) * p3
    score = ((t_0 + t_1) + t_2) ... + randint(1, 100) * 0.01

with `x ** e` == `float(x) ** float(e)` (libm pow) and each `x` one of the bounded state features of `FEATURES`.  The
library evaluates it with host-built power tables and separately rounded IEEE operations (spl_add_formula), so a formula
scores bit for bit as the Python expression does.  Register one in `HEURISTICS` and call `solve(heuristic_name=...)`:

    HEURISTICS['mine'] = Formula([(100, ('pts', 2.0)), (-1.5, ('saved', 0.5), ('cards', 1.0))])

`formula.reference()` is the same heuristic as a plain function of a reference `State`, for the reference's own
`HEURISTICS` (INTEGRATION.md).
"""
import math
import random

#: feature name -> (id of include/splendor_b200.h SPL_F_*, largest value; the domain is 0..largest)
FEATURES = {
    'pts': (0, 255), 'saved': (1, 65535), 'cards': (2, 90), 'gems': (3, 35), 'bonus': (4, 155),
    'resources': (5, 345), 'colors': (6, 5),
    **{f'gem_{c}': (7 + i, 7) for i, c in enumerate(('white', 'blue', 'green', 'red', 'black'))},
    **{f'bonus_{c}': (12 + i, 31) for i, c in enumerate(('white', 'blue', 'green', 'red', 'black'))},
}
MAX_TERMS = 8
MAX_FACTORS = 3


def feature_value(name: str, state) -> int:
    """The value of feature `name` on a state with fields cards, gems, bonus, pts, saved (this package's State or the
    reference's)."""
    if name == 'pts':
        return state.pts
    if name == 'saved':
        return state.saved
    if name == 'cards':
        return len(state.cards)
    if name == 'gems':
        return sum(state.gems)
    if name == 'bonus':
        return sum(state.bonus)
    if name == 'resources':
        return sum(state.gems) + 2 * sum(state.bonus)
    if name == 'colors':
        return sum(1 for b in state.bonus if b > 0)
    kind, colour = name.split('_')
    i = ('white', 'blue', 'green', 'red', 'black').index(colour)
    return state.gems[i] if kind == 'gem' else state.bonus[i]


class Formula:
    """An immutable, hashable formula heuristic: `Formula([(coef, (feature, exponent), ...), ...])`, 1 to 8 terms of 1 to
    3 factors.  Raises ValueError for an unknown feature, a negative or non-finite exponent, a non-finite coefficient,
    too many terms or factors, or a formula whose largest possible |t_0| + ... + |t_n| over the feature domains is not
    a finite double (its scores could be inf or NaN).

    Calling it scores one state on the GPU with solver.DEFAULT_NOISE, as the built-in HEURISTICS functions do."""

    __slots__ = ('terms', '_hash')

    def __init__(self, terms):
        norm = []
        for term in terms:
            term = tuple(term)
            if len(term) < 2:
                raise ValueError(f'formula term {term!r}: (coef, (feature, exponent), ...) with 1 to {MAX_FACTORS} factors')
            coef, factors = term[0], term[1:]
            if len(factors) > MAX_FACTORS:
                raise ValueError(f'formula term {term!r}: at most {MAX_FACTORS} factors')
            coef = float(coef)
            if not math.isfinite(coef):
                raise ValueError(f'formula term {term!r}: the coefficient is not finite')
            fs = []
            for f in factors:
                name, e = f
                if name not in FEATURES:
                    raise ValueError(f'formula term {term!r}: unknown feature {name!r} (known: {", ".join(FEATURES)})')
                e = float(e)
                if not math.isfinite(e) or e < 0:
                    raise ValueError(f'formula term {term!r}: exponent {e!r} is negative or not finite')
                fs.append((name, e + 0.0))
            norm.append((coef, *fs))
        if not 1 <= len(norm) <= MAX_TERMS:
            raise ValueError(f'a formula has 1 to {MAX_TERMS} terms, not {len(norm)}')
        bound = 0.0
        for coef, *fs in norm:
            t = abs(coef)
            for name, e in fs:
                try:
                    t *= float(FEATURES[name][1]) ** e  # pow does not decrease in x >= 0 for e >= 0
                except OverflowError:
                    t = math.inf
            bound += t
        if not math.isfinite(bound):
            raise ValueError('the largest possible |t_0| + ... + |t_n| of this formula over the feature domains is not a '
                             'finite double: its scores could be inf or NaN')
        object.__setattr__(self, 'terms', tuple(norm))
        object.__setattr__(self, '_hash', hash(self.terms))

    def __setattr__(self, name, value):
        raise AttributeError('Formula is immutable')

    def __eq__(self, other):
        return isinstance(other, Formula) and self.terms == other.terms

    def __hash__(self):
        return self._hash

    def __repr__(self):
        return f'Formula({list(self.terms)!r})'

    def terms_value(self, state) -> float:
        """t_0 + t_1 + ... (left to right) on `state`, without the noise term"""
        acc = None
        for coef, *fs in self.terms:
            t = coef
            for name, e in fs:
                t = t * float(feature_value(name, state)) ** e
            acc = t if acc is None else acc + t
        return acc

    def reference(self):
        """This heuristic as a plain-Python function of a reference `State` (fields cards, gems, bonus, pts, saved): the
        terms, then exactly one `random.randint(1, 100)` of the global generator, as the built-in heuristics draw it.
        Registered in the reference's own HEURISTICS, `random.seed(S)` + the unmodified reference reproduces
        `random.seed(S); State.solve(..., noise='mt')` of this package."""
        def heuristic(state) -> float:
            return self.terms_value(state) + random.randint(1, 100) * 0.01
        heuristic.__name__ = 'formula_heuristic'
        heuristic.__qualname__ = 'formula_heuristic'
        return heuristic

    def __call__(self, state) -> float:
        from .solver import _score_one
        return _score_one(self, state)

    def as_c(self):
        """the spl_formula struct of this formula (include/splendor_b200.h)"""
        from ._lib import Formula as CFormula
        f = CFormula()
        f.n_terms = len(self.terms)
        for i, (coef, *fs) in enumerate(self.terms):
            t = f.term[i]
            t.coef = coef
            t.n_factors = len(fs)
            for j, (name, e) in enumerate(fs):
                t.feature[j] = FEATURES[name][0]
                t.exponent[j] = e
        return f


#: the four built-in heuristics as formulas: bit-identical scores (src/solver.py:210-286)
BUILTIN_TWINS = {
    'simple': Formula([(1.0, ('saved', .4), ('pts', 2.5))]),
    'balanced': Formula([(100, ('pts', 2.8)), (10, ('saved', .5)), (5, ('resources', .3)), (3, ('cards', .6)),
                         (2, ('colors', .4))]),
    'aggressive': Formula([(200, ('pts', 3.2)), (5, ('saved', .3)), (2, ('bonus', .5))]),
    'efficiency': Formula([(50, ('pts', 2.0)), (30, ('saved', .7)), (20, ('bonus', 1.2)), (10, ('colors', .8))]),
}
