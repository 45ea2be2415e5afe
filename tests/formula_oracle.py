"""CPU oracle of formula heuristics: tests/formula_oracle.c (the oracle of oracle/, compiled as it is, plus formula
scoring and a formula-scored beam cut), built on first use into a temporary directory.  TEST INFRASTRUCTURE ONLY.

    score(states, formula, noise='const', draws=None)   the formula's score of every packed state
    Solver(goal_pts, formula, ...)                      oracle.Solver's level stepper, scored by the formula
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import oracle

_HERE = Path(__file__).resolve().parent
_SRC = _HERE / 'formula_oracle.c'
_ORACLE_SRC = _HERE.parent / 'oracle' / 'splendor_oracle.c'
_DECK = _HERE.parent / 'splendor-rl-gym_b200' / 'csrc' / 'deck_table.h'
# the oracle's own flags (oracle/Makefile): every * and + of a score rounds separately, as in CPython
CFLAGS = ['-O2', '-fPIC', '-std=gnu11', '-ffp-contract=off', '-shared']

FEATURE_IDS = {'pts': 0, 'saved': 1, 'cards': 2, 'gems': 3, 'bonus': 4, 'resources': 5, 'colors': 6,
               **{f'gem_{c}': 7 + i for i, c in enumerate(('white', 'blue', 'green', 'red', 'black'))},
               **{f'bonus_{c}': 12 + i for i, c in enumerate(('white', 'blue', 'green', 'red', 'black'))}}


class _Term(C.Structure):
    _fields_ = [('coef', C.c_double), ('n_factors', C.c_int32), ('feature', C.c_int32 * 3), ('exponent', C.c_double * 3)]


class _Formula(C.Structure):
    _fields_ = [('n_terms', C.c_int32), ('reserved', C.c_int32), ('term', _Term * 8)]


def cformula(formula) -> _Formula:
    """the oracle's struct of a formula: anything with `terms` ((coef, (feature, exponent), ...), ...)"""
    f = _Formula()
    f.n_terms = len(formula.terms)
    for i, (coef, *fs) in enumerate(formula.terms):
        f.term[i].coef = float(coef)
        f.term[i].n_factors = len(fs)
        for j, (name, e) in enumerate(fs):
            f.term[i].feature[j] = FEATURE_IDS[name]
            f.term[i].exponent[j] = float(e)
    return f


_lib = None


def lib():
    global _lib
    if _lib is None:
        h = hashlib.sha256(b''.join(p.read_bytes() for p in (_SRC, _ORACLE_SRC, _DECK))).hexdigest()[:16]
        so = Path(tempfile.gettempdir()) / f'splendor_formula_oracle_{os.getuid()}_{h}.so'
        if not so.exists():
            fd, tmp = tempfile.mkstemp(suffix='.so', dir=so.parent)
            os.close(fd)
            subprocess.run([os.environ.get('CC', 'gcc'), *CFLAGS, '-o', tmp, str(_SRC), '-lm'], check=True)
            os.replace(tmp, so)  # atomic: concurrent test processes never load a half-written library
        L = C.CDLL(str(so))
        L.orc_init.restype = C.c_int
        L.orcf_score.argtypes = [C.c_void_p, C.POINTER(_Formula), C.c_int, C.c_int]
        L.orcf_score.restype = C.c_double
        L.orc_solver_new.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int]
        L.orc_solver_new.restype = C.c_void_p
        L.orc_solver_free.argtypes = [C.c_void_p]
        L.orc_solver_set_identity.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_set_identity.restype = None
        L.orcf_solver_step.argtypes = [C.c_void_p, C.POINTER(_Formula), C.POINTER(oracle.LevelInfo)]
        L.orc_solver_nlevels.argtypes = [C.c_void_p]
        L.orc_solver_level_size.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_level_size.restype = C.c_int64
        L.orc_solver_level_states.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_level_states.restype = C.c_void_p
        L.orc_solver_level_links.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_level_links.restype = C.c_void_p
        L.orc_solver_path.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_init()
        _lib = L
    return _lib


def score(states: np.ndarray, formula, noise: str = 'const', draws=None) -> np.ndarray:
    """`draws`: the randint(1, 100) value of every state instead of `noise`"""
    states = np.ascontiguousarray(states)
    out = np.zeros(len(states), np.float64)
    f, nz, L = cformula(formula), oracle.NOISE_IDS[noise], lib()
    base, size = states.ctypes.data, oracle.STATE_DTYPE.itemsize
    for i in range(len(states)):
        out[i] = L.orcf_score(base + i * size, C.byref(f), nz, int(draws[i]) if draws is not None else 0)
    return out


class Solver:
    """oracle.Solver (same counters, levels and path) with the beam cut scored by `formula`"""

    def __init__(self, goal_pts, formula, *, beam_width=300_000, policy='stable', noise='const', identity='key'):
        root = oracle.pack_state((), (0,) * 5, (0,) * 5, 0, 0)
        self._f = cformula(formula)
        self._h = lib().orc_solver_new(root.ctypes.data, 1, goal_pts, 1, 0, beam_width, oracle.POLICY_IDS[policy],
                                       oracle.NOISE_IDS[noise])
        if identity != 'key':
            lib().orc_solver_set_identity(self._h, {'key': 0, 'pyhash': 1}[identity])
        self.infos = []
        self.done = False

    def step(self):
        li = oracle.LevelInfo()
        self.done = bool(lib().orcf_solver_step(self._h, C.byref(self._f), C.byref(li)))
        d = li.as_dict()
        self.infos.append(d)
        return d

    def run(self, max_levels=None):
        while not self.done:
            self.step()
            if max_levels is not None and len(self.infos) >= max_levels:
                break
        return self.infos

    @property
    def nlevels(self):
        return lib().orc_solver_nlevels(self._h)

    def level(self, i):
        """(states, links) of the queue at the top of while-iteration i (copies)"""
        n = lib().orc_solver_level_size(self._h, i)
        sp = lib().orc_solver_level_states(self._h, i)
        lp = lib().orc_solver_level_links(self._h, i)
        st = np.frombuffer((C.c_char * (n * oracle.STATE_DTYPE.itemsize)).from_address(sp), oracle.STATE_DTYPE).copy()
        lk = np.frombuffer((C.c_char * (n * 8)).from_address(lp), np.uint64).copy()
        return st, lk

    def path(self):
        out = np.zeros(self.nlevels, oracle.STATE_DTYPE)
        n = lib().orc_solver_path(self._h, out.ctypes.data, len(out))
        return out[:n]

    def close(self):
        if self._h:
            lib().orc_solver_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
