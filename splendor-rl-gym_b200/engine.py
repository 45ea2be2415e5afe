"""Host-side driver of the CUDA library: device buffers (torch), streams, and thin wrappers
over the C ABI (include/splendor_b200.h).  PyTorch is plumbing here -- it owns the caller-side
device tensors and the current stream; every computation happens inside libsplendor_b200.so.
"""
import ctypes as C

import numpy as np
import torch

from ._lib import Config, Key, LevelInfo, RGameInfo, check, lib

HEURISTIC_IDS = {'simple': 0, 'balanced': 1, 'aggressive': 2, 'efficiency': 3, 'competitive': 1}
TIE_IDS = {'stable': 0, 'det': 1, 'key': 1, 'det_ordered': 2}
IDENTITY_IDS = {'key': 0, 'pyhash': 1}
NOISE_IDS = {'const': 0, 'hash': 1, 'mt': 2}

M64 = (1 << 64) - 1


def heuristic_id(name: str) -> int:
    """Unknown names fall back to `simple`, as HEURISTICS.get(name, simple_heuristic) (src/solver.py:429)."""
    return HEURISTIC_IDS.get(name, 0)


# ------------------------------------------------------------------ packing (host side of spl_pack/spl_unpack)
def pack_key(cards, gems) -> int:
    m = 0
    for c in cards:
        m |= 1 << c
    g = 0
    for i, x in enumerate(gems):
        if not 0 <= x <= 7:
            raise ValueError(f'gem count out of range in {gems!r}')
        g |= x << (3 * i)
    return (m << 15) | g


def pack_aux(bonus, pts, saved) -> int:
    if not (0 <= saved < 1 << 16 and 0 <= pts < 1 << 8 and all(0 <= b < 32 for b in bonus)):
        raise ValueError('state fields out of the packed range (saved < 65536, pts < 256, bonus < 32)')
    a = saved | pts << 16
    for i, b in enumerate(bonus):
        a |= b << (24 + 5 * i)
    return a


def unpack_record(lo: int, hi: int, aux: int):
    k = (lo & M64) | (hi & M64) << 64
    gems = tuple((k >> (3 * i)) & 7 for i in range(5))
    m = (k >> 15) & ((1 << 90) - 1)
    cards = tuple(i for i in range(90) if (m >> i) & 1)
    bonus = tuple((aux >> (24 + 5 * i)) & 31 for i in range(5))
    return cards, bonus, gems, (aux >> 16) & 0xff, aux & 0xffff


class MTNoise:
    """The reference's own noise source: `random.randint(1, 100)` of Python's global Mersenne Twister
    (src/solver.py:4,215,247,260,284,810), drawn once per scored state in next_queue order.

    `random.randint(1, 100)` is `1 + _randbelow(100)`: take the top 7 bits of one 32-bit MT19937 output and
    retry while the value is >= 100.  The same stream is produced here in bulk with numpy's MT19937 bit
    generator started from `random.getstate()`; `finish()` leaves the global `random` module exactly
    where the reference would have left it."""

    def __init__(self):
        import random
        ver, state, gauss = random.getstate()
        self._ver, self._gauss = ver, gauss
        self._init = (np.array(state[:-1], dtype=np.uint32), int(state[-1]))
        self._bg = self._fresh()
        self._buf = np.zeros(0, np.uint8)   # accepted draws not handed out yet
        self._raw_at_buf_end = 0            # raw outputs consumed up to the end of the buffered draws
        self._raw_pos = np.zeros(0, np.int64)
        self.raw_used = 0                   # raw outputs the reference would have consumed so far

    def _fresh(self):
        bg = np.random.MT19937()
        bg.state = {'bit_generator': 'MT19937', 'state': {'key': self._init[0].copy(), 'pos': self._init[1]}}
        return bg

    def draw(self, n: int) -> np.ndarray:
        """the next n values of randint(1, 100) as uint8"""
        while len(self._buf) < n:
            m = max(1 << 16, int((n - len(self._buf)) * 1.4) + 1024)
            raw = self._bg.random_raw(m) >> 25
            ok = np.nonzero(raw < 100)[0]
            self._buf = np.concatenate([self._buf, (raw[ok] + 1).astype(np.uint8)])
            self._raw_pos = np.concatenate([self._raw_pos, ok + self._raw_at_buf_end + 1])
            self._raw_at_buf_end += m
        out, self._buf = self._buf[:n], self._buf[n:]
        if n:
            self.raw_used = int(self._raw_pos[n - 1])
        self._raw_pos = self._raw_pos[n:]
        return out

    def finish(self):
        """advance Python's global generator by exactly the outputs the reference would have consumed"""
        import random
        bg = self._fresh()
        left = self.raw_used
        while left > 0:
            step = min(left, 1 << 24)
            bg.random_raw(step)
            left -= step
        st = bg.state['state']
        random.setstate((self._ver, tuple(int(x) for x in st['key']) + (int(st['pos']),), self._gauss))


def _i64(x: int) -> int:
    x &= M64
    return x - (1 << 64) if x >> 63 else x


class _DevArray:
    """Zero-copy torch view of library-owned device memory (via __cuda_array_interface__)."""

    def __init__(self, ptr, shape, typestr='<i8'):
        self.__cuda_array_interface__ = {'shape': shape, 'typestr': typestr, 'data': (ptr, False), 'version': 3}


class Engine:
    """One CUDA context of the library on one device (spl_create / spl_destroy)."""

    _instances: dict = {}

    def __init__(self, device: int = 0, table_slots: int = 0, max_table_bytes: int = 0, chunk_parents: int = 0,
                 node_slots: int = 0, max_node_bytes: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError('splendor-rl-gym_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self.device = device
        self.tdev = torch.device('cuda', device)
        torch.cuda.init()
        with torch.cuda.device(device):
            torch.zeros(1, device=self.tdev)  # make sure the primary context exists
        cfg = Config(device, 0, table_slots, max_table_bytes, chunk_parents, node_slots, max_node_bytes)
        h = C.c_void_p()
        check(lib.spl_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.host_bytes = [0, 0]  # bytes this Python layer copied host->device / device->host itself (torch tensors)

    @classmethod
    def get(cls, device: int = 0, **kw) -> 'Engine':
        key = (device, tuple(sorted(kw.items())))
        if key not in cls._instances:
            cls._instances[key] = cls(device, **kw)
        return cls._instances[key]

    def close(self):
        if getattr(self, '_h', None):
            lib.spl_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -------------------------------------------------------------- helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.tdev).cuda_stream)

    def to_device(self, keys_np: np.ndarray, aux_np: np.ndarray):
        k = torch.from_numpy(np.ascontiguousarray(keys_np).view(np.int64).reshape(-1, 2)).to(self.tdev)
        a = torch.from_numpy(np.ascontiguousarray(aux_np).view(np.int64).reshape(-1)).to(self.tdev)
        return k, a

    def reset_visited(self):
        check(lib.spl_reset_visited(self._h, self._stream()), self._h)

    def set_identity(self, identity: str = 'key'):
        """Identity of the speedrun solver's visited set: 'key' = exact (cards, gems); 'pyhash' = the reference's
        own State.hash = hash((cards, gems)) (src/solver.py:316, :335-336), collisions merge as in its dict."""
        check(lib.spl_set_identity(self._h, IDENTITY_IDS[identity]), self._h)

    def set_link_budget(self, device_bytes: int = 0):
        """Device bytes the next solvers may hold in parent-link columns (trail, src/solver.py:449, :459-464) before the
        oldest levels spill to pinned host memory; 0 = keep everything on the device."""
        check(lib.spl_set_link_budget(self._h, int(device_bytes)), self._h)

    def spilled_bytes(self) -> int:
        n = C.c_int64()
        check(lib.spl_spilled_bytes(self._h, C.byref(n)), self._h)
        return n.value

    def pyhash(self, keys: torch.Tensor) -> torch.Tensor:
        """hash((cards, gems)) per key (src/solver.py:316), int64 view of CPython's value"""
        out = torch.empty(keys.shape[0], dtype=torch.int64, device=self.tdev)
        check(lib.spl_pyhash(self._h, keys.data_ptr(), keys.shape[0], out.data_ptr(), self._stream()), self._h)
        return out

    def visited_count(self) -> int:
        n = C.c_int64()
        check(lib.spl_visited_count(self._h, C.byref(n)), self._h)
        return n.value

    def launch_count(self) -> int:
        n = C.c_int64()
        check(lib.spl_launch_count(self._h, C.byref(n)), self._h)
        return n.value

    def transfer_bytes(self):
        """(host->device, device->host) bytes copied so far: by the library (spl_transfer_bytes) plus by this layer"""
        a, b = C.c_int64(), C.c_int64()
        check(lib.spl_transfer_bytes(self._h, C.byref(a), C.byref(b)), self._h)
        return a.value + self.host_bytes[0], b.value + self.host_bytes[1]

    # -------------------------------------------------------------- stage operators
    def expand(self, keys: torch.Tensor, aux: torch.Tensor):
        """State.__iter__ for a batch (src/solver.py:357-388) -> (cand_keys [m,2], cand_aux [m], cand_link [m])."""
        n = keys.shape[0]
        cap = max(64, n * 40)
        while True:
            ck = torch.empty((cap, 2), dtype=torch.int64, device=self.tdev)
            ca = torch.empty(cap, dtype=torch.int64, device=self.tdev)
            cl = torch.empty(cap, dtype=torch.int64, device=self.tdev)
            m = C.c_int64()
            rc = lib.spl_expand(self._h, keys.data_ptr(), aux.data_ptr(), n, ck.data_ptr(), ca.data_ptr(),
                                cl.data_ptr(), cap, C.byref(m), self._stream())
            if rc == -6:  # SPL_E_CAPACITY: m holds the needed size
                cap = m.value
                continue
            check(rc, self._h)
            return ck[:m.value], ca[:m.value], cl[:m.value]

    def dedup(self, cand_keys: torch.Tensor, cand_aux: torch.Tensor):
        """First-arrival dedup against the context's visited set (src/solver.py:447-450)."""
        n = cand_keys.shape[0]
        uk = torch.empty((max(n, 1), 2), dtype=torch.int64, device=self.tdev)
        ua = torch.empty(max(n, 1), dtype=torch.int64, device=self.tdev)
        us = torch.empty(max(n, 1), dtype=torch.int64, device=self.tdev)
        m = C.c_int64()
        check(lib.spl_dedup(self._h, cand_keys.data_ptr(), cand_aux.data_ptr(), n, uk.data_ptr(), ua.data_ptr(),
                            us.data_ptr(), C.byref(m), self._stream()), self._h)
        return uk[:m.value], ua[:m.value], us[:m.value]

    def score(self, heuristic: str, keys: torch.Tensor, aux: torch.Tensor, noise: str = 'const') -> torch.Tensor:
        n = keys.shape[0]
        out = torch.empty(n, dtype=torch.float64, device=self.tdev)
        check(lib.spl_score(self._h, heuristic_id(heuristic), NOISE_IDS[noise], keys.data_ptr(), aux.data_ptr(), n,
                            out.data_ptr(), self._stream()), self._h)
        return out

    def topk(self, scores: torch.Tensor, keys: torch.Tensor, k: int, tie: str = 'stable') -> torch.Tensor:
        n = scores.shape[0]
        out = torch.empty(max(min(n, k), 1), dtype=torch.int64, device=self.tdev)
        m = C.c_int64()
        check(lib.spl_topk(self._h, scores.data_ptr(), keys.data_ptr(), n, k, TIE_IDS[tie], out.data_ptr(),
                           C.byref(m), self._stream()), self._h)
        return out[:m.value]

    # -------------------------------------------------------------- realistic mode (MultiPlayerState)
    def rexpand(self, rcfg, recs_np: np.ndarray) -> np.ndarray:
        """MultiPlayerState.__iter__ for a batch of 96-byte records (host numpy in, host numpy out)."""
        recs_np = np.ascontiguousarray(recs_np).reshape(-1)
        n = len(recs_np)
        src = torch.from_numpy(recs_np.view(np.uint8).reshape(n, 96).copy()).to(self.tdev)
        cap = max(64, n * 27)
        out = torch.empty((cap, 96), dtype=torch.uint8, device=self.tdev)
        m = C.c_int64()
        check(lib.spl_rexpand(self._h, C.byref(rcfg), src.data_ptr(), n, out.data_ptr(), cap, C.byref(m), self._stream()),
              self._h)
        return out[:m.value].cpu().numpy().reshape(-1).view(recs_np.dtype).copy()

    def rscore(self, rcfg, recs_np: np.ndarray) -> np.ndarray:
        recs_np = np.ascontiguousarray(recs_np).reshape(-1)
        n = len(recs_np)
        src = torch.from_numpy(recs_np.view(np.uint8).reshape(n, 96).copy()).to(self.tdev)
        out = torch.empty(n, dtype=torch.float64, device=self.tdev)
        check(lib.spl_rscore(self._h, C.byref(rcfg), src.data_ptr(), n, out.data_ptr(), self._stream()), self._h)
        return out.cpu().numpy()

    def rpack(self, rcfg, recs_np: np.ndarray) -> np.ndarray:
        """exact 384-bit identity keys (6 x uint64 per record) of a batch of realistic-mode records"""
        recs_np = np.ascontiguousarray(recs_np).reshape(-1)
        n = len(recs_np)
        src = torch.from_numpy(recs_np.view(np.uint8).reshape(n, 96).copy()).to(self.tdev)
        out = torch.zeros((n, 6), dtype=torch.int64, device=self.tdev)
        check(lib.spl_rpack(self._h, C.byref(rcfg), src.data_ptr(), n, out.data_ptr(), self._stream()), self._h)
        return out.cpu().numpy().view(np.uint64)

    def rsolver(self, rcfg, root_rec_np: np.ndarray, beam_width: int, keep_links: bool = True) -> 'RLevelSolver':
        return RLevelSolver(self, rcfg, root_rec_np, beam_width, keep_links)

    def rbatch_solver(self, rcfgs, roots_np: np.ndarray, beams, keep_links: bool = True) -> 'RBatchSolver':
        """spl_rbatch_create: len(rcfgs) realistic-mode games searched in lockstep (root record and beam width per game)."""
        return RBatchSolver(self, rcfgs, roots_np, beams, keep_links)

    def sbatch_solver(self, roots_np: np.ndarray, goals, use_heuristic, heuristics, beams, tie: str = 'stable',
                      noise: str = 'const', keep_links: bool = True) -> 'SBatchSolver':
        """spl_sbatch_create: len(roots_np) speedrun games searched in lockstep.  roots_np: 32-byte rows {lo, hi, aux,
        link} (an [n, 4] uint64 array); goals, use_heuristic, heuristics (names or ids) and beams: one per game."""
        return SBatchSolver(self, roots_np, goals, use_heuristic, heuristics, beams, tie, noise, keep_links)

    # -------------------------------------------------------------- fused solver
    def solver(self, root_key: int, root_aux: int, goal_pts: int, use_heuristic: bool, heuristic: str, beam_width: int,
               tie: str = 'stable', noise: str = 'const', keep_links: bool = True, identity: str = 'key',
               queue: np.ndarray = None) -> 'LevelSolver':
        """With `queue` (an array of 32-byte rows {lo, hi, aux, link} in rank order; links ignored) the solve starts
        from that level-0 queue instead of the one state (root_key, root_aux), which are then ignored."""
        self.set_identity(identity)
        return LevelSolver(self, root_key, root_aux, goal_pts, use_heuristic, heuristic, beam_width, tie, noise,
                           keep_links, queue)


class Stepper:
    """run() of the level solvers: step() is one `while queue` iteration that appends its counters to self.infos"""

    def run(self, max_levels=None):
        while not self.ended:
            self.step()
            if max_levels is not None and len(self.infos) >= max_levels:
                break
        return self.infos


class LevelSolver(Stepper):
    """spl_solver_*: one object per solve(); step() == one `while queue` iteration (src/solver.py:434-457)."""

    def __init__(self, eng: Engine, root_key, root_aux, goal_pts, use_heuristic, heuristic, beam_width, tie, noise,
                 keep_links, queue=None):
        self.eng = eng
        h = C.c_void_p()
        args = (goal_pts, int(bool(use_heuristic)), heuristic_id(heuristic), beam_width, TIE_IDS[tie], NOISE_IDS[noise],
                int(keep_links), C.byref(h))
        if queue is None:
            k = Key(root_key & M64, root_key >> 64)
            check(lib.spl_solver_create(eng._h, C.byref(k), root_aux, *args), eng._h)
        else:
            rows = np.ascontiguousarray(queue)
            if rows.dtype.itemsize != 32:
                raise ValueError(f'queue rows must be 32 bytes {{lo, hi, aux, link}}, not {rows.dtype}')
            check(lib.spl_solver_create_queue(eng._h, rows.ctypes.data, len(rows), *args), eng._h)
        self._h = h
        self.infos = []
        self.ended = False
        self.noise_source = MTNoise() if noise == 'mt' else None

    def step(self) -> dict:
        li = LevelInfo()
        check(lib.spl_solver_step(self._h, C.byref(li), self.eng._stream()), self.eng._h)
        if li.kept == -1 and not li.ended:  # noise='mt': hand the level its randint draws (arrival order)
            if self.noise_source is None:
                raise RuntimeError("solver created with noise='mt' needs a noise_source")
            draws = torch.from_numpy(self.noise_source.draw(li.unique)).to(self.eng.tdev)
            check(lib.spl_solver_cut(self._h, draws.data_ptr(), li.unique, C.byref(li), self.eng._stream()), self.eng._h)
        d = li.as_dict()
        self.infos.append(d)
        self.ended = bool(li.ended)
        return d

    def frontier(self) -> torch.Tensor:
        """Current queue as an int64 tensor [n, 4] = (lo, hi, aux, link) viewing library memory."""
        kp, n = C.c_void_p(), C.c_int64()
        check(lib.spl_solver_frontier(self._h, C.byref(kp), None, None, C.byref(n)), self.eng._h)
        if n.value == 0:
            return torch.empty((0, 4), dtype=torch.int64, device=self.eng.tdev)
        return torch.as_tensor(_DevArray(kp.value, (n.value, 4)), device=self.eng.tdev)

    def path(self):
        """(ranks, ordinals): ordinals[i] indexes list(iter(path[i])) to give path[i+1] (src/solver.py:459-464)."""
        cap = len(self.infos) + 2
        ranks = (C.c_int64 * cap)()
        ords = (C.c_int32 * cap)()
        nm = C.c_int32()
        check(lib.spl_solver_path(self._h, ranks, ords, cap, C.byref(nm)), self.eng._h)
        return list(ranks[:nm.value + 1]), list(ords[:nm.value])

    def close(self):
        if getattr(self, '_h', None):
            lib.spl_solver_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RLevelSolver(LevelSolver):
    """spl_rsolver_create + spl_solver_step: one object per MultiPlayerState.solve()."""

    def __init__(self, eng: Engine, rcfg, root_rec_np, beam_width, keep_links):
        self.eng = eng
        root = np.ascontiguousarray(root_rec_np).reshape(-1)[:1].copy()
        h = C.c_void_p()
        check(lib.spl_rsolver_create(eng._h, C.byref(rcfg), root.ctypes.data, beam_width, int(keep_links), C.byref(h)), eng._h)
        self._h = h
        self._dtype = root.dtype
        self.infos = []
        self.ended = False
        self.noise_source = MTNoise() if rcfg.noise == 2 else None

    def progress(self, rcfg, running_max: int):
        """(rank, record, max pts) of every queued state that raises the running maximum of max-player-points
        while the queue is scanned in order, up to the first finished game (src/solver.py:825-836)."""
        p, n = C.c_void_p(), C.c_int64()
        check(lib.spl_rsolver_frontier(self._h, C.byref(p), C.byref(n)), self.eng._h)
        if n.value == 0:
            return []
        mp = torch.empty(n.value, dtype=torch.uint8, device=self.eng.tdev)
        check(lib.spl_rmaxpts(self.eng._h, C.byref(rcfg), p.value, n.value, mp.data_ptr(), self.eng._stream()), self.eng._h)
        mp = mp.to(torch.int64)
        run = torch.cummax(mp, 0).values
        prev = torch.clamp(torch.cat([torch.full((1,), running_max, dtype=torch.int64, device=mp.device), run[:-1]]), min=running_max)
        hits = torch.nonzero(mp > prev).flatten().tolist()
        if not hits:
            return []
        recs = torch.as_tensor(_DevArray(p.value, (n.value, 96), '|u1'), device=self.eng.tdev)
        sel = recs[torch.tensor(hits, device=self.eng.tdev)].cpu().numpy().reshape(-1).view(self._dtype)
        return [(h, sel[i], int(mp[h])) for i, h in enumerate(hits)]

    def frontier_size(self) -> int:
        p, n = C.c_void_p(), C.c_int64()
        check(lib.spl_rsolver_frontier(self._h, C.byref(p), C.byref(n)), self.eng._h)
        return n.value

    def frontier(self) -> np.ndarray:
        """current queue as host records (96 B each)"""
        p, n = C.c_void_p(), C.c_int64()
        check(lib.spl_rsolver_frontier(self._h, C.byref(p), C.byref(n)), self.eng._h)
        if n.value == 0:
            return np.zeros(0, self._dtype)
        t = torch.as_tensor(_DevArray(p.value, (n.value, 96), '|u1'), device=self.eng.tdev)
        return t.cpu().numpy().reshape(-1).view(self._dtype).copy()


class RBatchSolver(Stepper):
    """spl_rbatch_create + spl_solver_step: B MultiPlayerState.solve() searches in lockstep (realistic.solve_many)."""

    def __init__(self, eng: Engine, rcfgs, roots_np, beams, keep_links=True):
        self.eng = eng
        self.n_games = len(rcfgs)
        roots = np.ascontiguousarray(roots_np).reshape(-1)
        if len(roots) != self.n_games or len(beams) != self.n_games:
            raise ValueError(f'{self.n_games} configs, {len(roots)} roots and {len(beams)} beam widths')
        cfgs = (type(rcfgs[0]) * self.n_games)(*rcfgs)
        bw = np.ascontiguousarray(beams, dtype=np.int64)
        h = C.c_void_p()
        check(lib.spl_rbatch_create(eng._h, cfgs, roots.ctypes.data, bw.ctypes.data, self.n_games, int(keep_links),
                                    C.byref(h)), eng._h)
        self._h = h
        self._dtype = roots.dtype
        self.infos = []
        self.ended = False

    def step(self) -> dict:
        """One level of every running game: the aggregate counters (spl_level_info) plus 'games', the per-game
        counters (a game's dict stops changing once it has ended)."""
        li = LevelInfo()
        check(lib.spl_solver_step(self._h, C.byref(li), self.eng._stream()), self.eng._h)
        d = li.as_dict()
        d['games'] = self.games()
        self.infos.append(d)
        self.ended = bool(li.ended)
        return d

    def games(self) -> list:
        out = (RGameInfo * self.n_games)()
        check(lib.spl_rbatch_games(self._h, out, self.n_games), self.eng._h)
        return [g.as_dict() for g in out]

    def frontier(self, game: int) -> np.ndarray:
        """game `game`'s current queue as host records (96 B each); empty once the game has ended"""
        p, n = C.c_void_p(), C.c_int64()
        check(lib.spl_rbatch_frontier(self._h, int(game), C.byref(p), C.byref(n)), self.eng._h)
        if n.value == 0:
            return np.zeros(0, self._dtype)
        t = torch.as_tensor(_DevArray(p.value, (n.value, 96), '|u1'), device=self.eng.tdev)
        return t.cpu().numpy().reshape(-1).view(self._dtype).copy()

    def lines(self) -> list:
        """every game's line as host records, root first (spl_rbatch_lines)"""
        plies = (C.c_int32 * self.n_games)()
        cap = max((g['level'] for g in self.games()), default=0) + 1
        recs = np.zeros(self.n_games * cap, self._dtype)
        check(lib.spl_rbatch_lines(self._h, recs.ctypes.data, cap, plies), self.eng._h)
        return [recs[g * cap:g * cap + plies[g] + 1] for g in range(self.n_games)]

    def close(self):
        if getattr(self, '_h', None):
            lib.spl_solver_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class SBatchSolver(Stepper):
    """spl_sbatch_create + spl_solver_step: B State.solve() searches in lockstep (State.solve_many)."""

    def __init__(self, eng: Engine, roots_np, goals, use_heuristic, heuristics, beams, tie='stable', noise='const',
                 keep_links=True):
        self.eng = eng
        roots = np.ascontiguousarray(roots_np, dtype=np.uint64).reshape(-1, 4)
        self.n_games = len(roots)
        cols = [goals, use_heuristic, heuristics, beams]
        if any(len(x) != self.n_games for x in cols):
            raise ValueError(f'{self.n_games} roots, but {[len(x) for x in cols]} goals / kinds / heuristics / beam widths')
        ids = [h if isinstance(h, int) else heuristic_id(h) for h in heuristics]
        g = np.ascontiguousarray(goals, dtype=np.int32)
        u = np.ascontiguousarray([int(bool(x)) for x in use_heuristic], dtype=np.int32)
        h = np.ascontiguousarray(ids, dtype=np.int32)
        bw = np.ascontiguousarray(beams, dtype=np.int64)
        hd = C.c_void_p()
        check(lib.spl_sbatch_create(eng._h, roots.ctypes.data, g.ctypes.data, u.ctypes.data, h.ctypes.data, bw.ctypes.data,
                                    self.n_games, TIE_IDS[tie], NOISE_IDS[noise], int(keep_links), C.byref(hd)), eng._h)
        self._h = hd
        self.infos = []
        self.ended = False

    def step(self) -> dict:
        """One level of every running game: the aggregate counters (spl_level_info) plus 'games', the per-game
        counters (a game's dict stops changing once it has ended)."""
        li = LevelInfo()
        check(lib.spl_solver_step(self._h, C.byref(li), self.eng._stream()), self.eng._h)
        d = li.as_dict()
        d['games'] = self.games()
        self.infos.append(d)
        self.ended = bool(li.ended)
        return d

    def games(self) -> list:
        out = (RGameInfo * self.n_games)()
        check(lib.spl_sbatch_games(self._h, out, self.n_games), self.eng._h)
        return [g.as_dict() for g in out]

    def frontier(self, game: int) -> np.ndarray:
        """game `game`'s current queue as host rows [n, 4] uint64 (lo, hi, aux, link); empty once the game has ended"""
        p, n = C.c_void_p(), C.c_int64()
        check(lib.spl_sbatch_frontier(self._h, int(game), C.byref(p), C.byref(n)), self.eng._h)
        if n.value == 0:
            return np.zeros((0, 4), np.uint64)
        return torch.as_tensor(_DevArray(p.value, (n.value, 4)), device=self.eng.tdev).cpu().numpy().view(np.uint64)

    def lines(self) -> list:
        """every game's line as host rows [plies + 1, 4] uint64, root first (spl_sbatch_lines)"""
        plies = (C.c_int32 * self.n_games)()
        cap = max((g['level'] for g in self.games()), default=0) + 1
        rows = np.zeros((self.n_games * cap, 4), np.uint64)
        check(lib.spl_sbatch_lines(self._h, rows.ctypes.data, cap, plies), self.eng._h)
        return [rows[g * cap:g * cap + plies[g] + 1] for g in range(self.n_games)]

    def close(self):
        if getattr(self, '_h', None):
            lib.spl_solver_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
