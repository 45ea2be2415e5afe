"""ctypes front-end of the CPU oracle (oracle/splendor_oracle.c).  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / `--impl reference`
legs may import this package; the product package (splendor-rl-gym_b200/) never does.
"""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
_LIB = _HERE / '_build' / 'liboracle.so'

STATE_DTYPE = np.dtype([('lo', '<u8'), ('hi', '<u8'), ('aux', '<u8')])
HEURISTIC_IDS = {'simple': 0, 'balanced': 1, 'aggressive': 2, 'efficiency': 3, 'competitive': 1}
POLICY_IDS = {'stable': 0, 'det': 1}
NOISE_IDS = {'const': 0, 'hash': 1}


class LevelInfo(C.Structure):
    _fields_ = [('level', C.c_int32), ('frontier', C.c_int64), ('expanded', C.c_int64),
                ('generated', C.c_int64), ('unique', C.c_int64), ('kept', C.c_int64),
                ('goal_rank', C.c_int64), ('visited', C.c_int64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def build(force: bool = False) -> Path:
    src = _HERE / 'splendor_oracle.c'
    if force or not _LIB.exists() or _LIB.stat().st_mtime < src.stat().st_mtime:
        subprocess.run(['make', '-C', str(_HERE), '-s'], check=True)
    return _LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(str(_LIB))
        L.orc_init.restype = C.c_int
        L.orc_take_gems.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_buys.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_subtract_with_bonus.argtypes = [C.c_void_p] * 4
        L.orc_expand.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_score.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.orc_score.restype = C.c_double
        L.orc_solver_new.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int]
        L.orc_solver_new.restype = C.c_void_p
        L.orc_solver_free.argtypes = [C.c_void_p]
        L.orc_solver_set_identity.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_set_identity.restype = None
        L.orc_pyhash.argtypes = [C.c_void_p]
        L.orc_pyhash.restype = C.c_uint64
        L.orc_solver_step.argtypes = [C.c_void_p, C.POINTER(LevelInfo)]
        L.orc_solver_nlevels.argtypes = [C.c_void_p]
        L.orc_solver_level_size.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_level_size.restype = C.c_int64
        L.orc_solver_level_states.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_level_states.restype = C.c_void_p
        L.orc_solver_level_links.argtypes = [C.c_void_p, C.c_int]
        L.orc_solver_level_links.restype = C.c_void_p
        L.orc_solver_goal_rank.argtypes = [C.c_void_p]
        L.orc_solver_goal_rank.restype = C.c_int64
        L.orc_solver_path.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.orc_takes_of.argtypes = [C.c_uint, C.c_void_p]
        L.orc_init()
        _lib = L
    return _lib


# ---------------------------------------------------------------- packing helpers (oracle-side)
def pack_state(cards, bonus, gems, pts, saved) -> np.ndarray:
    m = 0
    for c in cards:
        m |= 1 << c
    g = 0
    for i, x in enumerate(gems):
        g |= x << (3 * i)
    k = (m << 15) | g
    aux = (saved & 0xffff) | (pts & 0xff) << 16
    for i, b in enumerate(bonus):
        aux |= (b & 31) << (24 + 5 * i)
    s = np.zeros(1, STATE_DTYPE)
    s['lo'] = k & ((1 << 64) - 1)
    s['hi'] = k >> 64
    s['aux'] = aux
    return s


def unpack_state(rec):
    k = int(rec['lo']) | int(rec['hi']) << 64
    aux = int(rec['aux'])
    gems = tuple((k >> (3 * i)) & 7 for i in range(5))
    m = k >> 15
    cards = tuple(i for i in range(90) if (m >> i) & 1)
    bonus = tuple((aux >> (24 + 5 * i)) & 31 for i in range(5))
    return dict(cards=cards, bonus=bonus, gems=gems, pts=(aux >> 16) & 0xff, saved=aux & 0xffff, key=k)


def take_gems(g):
    a = np.array(g, np.uint8)
    out = np.zeros((128, 5), np.uint8)
    n = lib().orc_take_gems(a.ctypes.data, out.ctypes.data)
    return [tuple(int(x) for x in r) for r in out[:n]]


def buys(key):
    a = np.array(key, np.uint8)
    out = np.zeros(90, np.uint8)
    n = lib().orc_buys(a.ctypes.data, out.ctypes.data)
    return [int(x) for x in out[:n]]


def subtract_with_bonus(gems, cost, bonus):
    g, c, b = (np.array(x, np.uint8) for x in (gems, cost, bonus))
    out = np.zeros(5, np.uint8)
    saved = lib().orc_subtract_with_bonus(g.ctypes.data, c.ctypes.data, b.ctypes.data, out.ctypes.data)
    return tuple(int(x) for x in out), saved


def expand(state_rec: np.ndarray) -> np.ndarray:
    out = np.zeros(192, STATE_DTYPE)
    s = np.ascontiguousarray(state_rec).reshape(1)
    n = lib().orc_expand(s.ctypes.data, out.ctypes.data)
    return out[:n].copy()


def pyhash(states: np.ndarray) -> np.ndarray:
    """hash((cards, gems)) of src/solver.py:316 as an unsigned 64-bit value, per packed state"""
    states = np.ascontiguousarray(states)
    out = np.zeros(len(states), np.uint64)
    base = states.ctypes.data
    L = lib()
    for i in range(len(states)):
        out[i] = L.orc_pyhash(base + i * STATE_DTYPE.itemsize)
    return out


def score(states: np.ndarray, heuristic: str, noise: str = 'const') -> np.ndarray:
    states = np.ascontiguousarray(states)
    out = np.zeros(len(states), np.float64)
    h, nz = HEURISTIC_IDS.get(heuristic, 0), NOISE_IDS[noise]
    base = states.ctypes.data
    L = lib()
    for i in range(len(states)):
        out[i] = L.orc_score(base + i * STATE_DTYPE.itemsize, h, nz)
    return out


class Solver:
    """Level stepper over the oracle's restatement of State.solve (src/solver.py:390-464).  `root`: the packed
    state(s) of level 0 in rank order (fields lo, hi, aux; others ignored), each registered as visited."""

    def __init__(self, goal_pts=15, *, use_heuristic=False, heuristic_name='simple', beam_width=300_000,
                 policy='stable', noise='const', root=None, identity='key'):
        if root is None:
            root = pack_state((), (0,) * 5, (0,) * 5, 0, 0)
        root = np.asarray(root).reshape(-1)
        if len(root) < 1:
            raise ValueError('the level-0 queue needs at least one state')
        self._root = np.zeros(len(root), STATE_DTYPE)
        for f in ('lo', 'hi', 'aux'):
            self._root[f] = root[f]
        self._h = lib().orc_solver_new(self._root.ctypes.data, len(self._root), goal_pts, int(use_heuristic),
                                       HEURISTIC_IDS.get(heuristic_name, 0), beam_width,
                                       POLICY_IDS[policy], NOISE_IDS[noise])
        if identity != 'key':  # 'pyhash': dedup on the reference's own 64-bit hash((cards, gems))
            lib().orc_solver_set_identity(self._h, {'key': 0, 'pyhash': 1}[identity])
        self.infos = []
        self.done = False

    def step(self):
        li = LevelInfo()
        self.done = bool(lib().orc_solver_step(self._h, C.byref(li)))
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
        """(states, links) of the queue at the top of while-iteration i (copies)."""
        n = lib().orc_solver_level_size(self._h, i)
        sp = lib().orc_solver_level_states(self._h, i)
        lp = lib().orc_solver_level_links(self._h, i)
        st = np.frombuffer((C.c_char * (n * STATE_DTYPE.itemsize)).from_address(sp), STATE_DTYPE).copy()
        lk = np.frombuffer((C.c_char * (n * 8)).from_address(lp), np.uint64).copy()
        return st, lk

    def path(self):
        out = np.zeros(self.nlevels, STATE_DTYPE)
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


# ================================================================ realistic mode (MultiPlayerState)
RPLAYER_DTYPE = np.dtype([('mlo', '<u8'), ('mhi', '<u4'), ('gems', '<u2'), ('saved', '<u2')])
RREC_DTYPE = np.dtype([('p', RPLAYER_DTYPE, (4,)), ('vis', 'u1', (12,)), ('cur', 'u1'), ('pad', 'u1', (3,)),
                       ('link', '<u8'), ('spare', '<u8')])
assert RREC_DTYPE.itemsize == 96


class RConfig(C.Structure):
    _fields_ = [('num_players', C.c_int32), ('target_points', C.c_int32), ('gems_per_color', C.c_int32),
                ('noise_mode', C.c_int32), ('deck_len', C.c_int32 * 3), ('deck', (C.c_uint8 * 40) * 3)]


def make_rconfig(num_players, target_points, gems_per_color, tiers, noise='const') -> RConfig:
    """tiers = three full card sequences (visible cards first), as CardMarket.from_full_deck builds them."""
    cfg = RConfig(num_players, target_points, gems_per_color, NOISE_IDS[noise])
    for t, seq in enumerate(tiers):
        cfg.deck_len[t] = len(seq)
        for i, c in enumerate(seq):
            cfg.deck[t][i] = c
    return cfg


def rident_bytes(rec, num_players) -> bytes:
    """canonical identity bytes of one record (what tests/golden/make_golden.py::rrec_bytes hashes)"""
    return rec['p'][:num_players].tobytes() + rec['vis'].tobytes() + bytes([int(rec['cur'])])


def _rlib():
    L = lib()
    if not getattr(L, '_r_ready', False):
        L.orc_r_root.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_r_expand.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.orc_r_score.argtypes = [C.c_void_p, C.c_void_p]
        L.orc_r_score.restype = C.c_double
        L.orc_r_pts.argtypes = [C.c_void_p, C.c_int]
        L.orc_rsolver_new.argtypes = [C.c_void_p, C.c_int64]
        L.orc_rsolver_new.restype = C.c_void_p
        L.orc_rsolver_free.argtypes = [C.c_void_p]
        L.orc_rsolver_step.argtypes = [C.c_void_p, C.POINTER(LevelInfo)]
        L.orc_rsolver_nlevels.argtypes = [C.c_void_p]
        L.orc_rsolver_level_size.argtypes = [C.c_void_p, C.c_int]
        L.orc_rsolver_level_size.restype = C.c_int64
        L.orc_rsolver_level_states.argtypes = [C.c_void_p, C.c_int]
        L.orc_rsolver_level_states.restype = C.c_void_p
        L.orc_rsolver_goal_rank.argtypes = [C.c_void_p]
        L.orc_rsolver_goal_rank.restype = C.c_int64
        L.orc_rsolver_smin.argtypes = [C.c_void_p]
        L.orc_rsolver_smin.restype = C.c_double
        L.orc_rsolver_smax.argtypes = [C.c_void_p]
        L.orc_rsolver_smax.restype = C.c_double
        L.orc_rsolver_path.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L._r_ready = True
    return L


def r_root(cfg: RConfig) -> np.ndarray:
    out = np.zeros(1, RREC_DTYPE)
    _rlib().orc_r_root(C.byref(cfg), out.ctypes.data)
    return out


def r_expand(cfg: RConfig, rec: np.ndarray) -> np.ndarray:
    out = np.zeros(32, RREC_DTYPE)
    s = np.ascontiguousarray(rec).reshape(1)
    n = _rlib().orc_r_expand(C.byref(cfg), s.ctypes.data, out.ctypes.data)
    return out[:n].copy()


def r_score(cfg: RConfig, recs: np.ndarray) -> np.ndarray:
    recs = np.ascontiguousarray(recs)
    L = _rlib()
    return np.array([L.orc_r_score(C.byref(cfg), recs.ctypes.data + i * 96) for i in range(len(recs))], np.float64)


def r_pts(rec, player) -> int:
    s = np.ascontiguousarray(rec).reshape(1)
    return _rlib().orc_r_pts(s.ctypes.data, player)


class RSolver:
    """Level stepper over the oracle's restatement of MultiPlayerState.solve (src/solver.py:750-860)."""

    def __init__(self, cfg: RConfig, beam_width=20_000):
        self.cfg = cfg
        self._h = _rlib().orc_rsolver_new(C.byref(cfg), beam_width)
        self.infos, self.done = [], False

    def step(self):
        li = LevelInfo()
        self.done = bool(_rlib().orc_rsolver_step(self._h, C.byref(li)))
        self.infos.append(li.as_dict())
        return self.infos[-1]

    def run(self):
        while not self.done:
            self.step()
        return self.infos

    @property
    def nlevels(self):
        return _rlib().orc_rsolver_nlevels(self._h)

    def level(self, i):
        n = _rlib().orc_rsolver_level_size(self._h, i)
        sp = _rlib().orc_rsolver_level_states(self._h, i)
        return np.frombuffer((C.c_char * (n * 96)).from_address(sp), RREC_DTYPE).copy()

    def path(self):
        out = np.zeros(self.nlevels, RREC_DTYPE)
        n = _rlib().orc_rsolver_path(self._h, out.ctypes.data, len(out))
        return out[:n]

    def score_range(self):
        return _rlib().orc_rsolver_smin(self._h), _rlib().orc_rsolver_smax(self._h)

    def close(self):
        if self._h:
            _rlib().orc_rsolver_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
