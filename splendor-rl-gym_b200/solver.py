"""Speedrun solver front-end: the reference's `State` / `HEURISTICS` / `solve()` surface
(src/solver.py:207-464) driven by the CUDA library.

What runs where
  * `State.solve()`      -> spl_solver_* (expand + dedup + score + top-k kernels, one level per step)
  * `State.solve_many()` -> spl_sbatch_* (many searches in lockstep on one GPU, lines rebuilt on the device)
  * `State.__iter__()`   -> spl_expand on a batch of one
  * `HEURISTICS[name]()` -> spl_score on a batch of one
  * path reconstruction  -> spl_solver_path (parent ranks + ordinals), replayed through `__iter__`
There is no CPU implementation of the search in this package.

Tie-break / noise policy (SURVEY.md 8a-N).  The reference adds `randint(1, 100) * 0.01` drawn
from the unseeded global Mersenne Twister to every score, so it is not reproducible against
itself.  This path replaces the draw by a declared deterministic source:
  noise='const' : randint -> 50            noise='hash' : randint -> 1 + splitmix64(key) % 100
  noise='mt'    : the reference's own stream -- Python's global Mersenne Twister, one randint(1, 100)
                  per scored state in next_queue order; `random.seed(S); solve(..., noise='mt')` then
                  reproduces `random.seed(S)` + the UNMODIFIED reference (any number of GPUs: every rank
                  replays the same stream and indexes it by global arrival order)
and breaks score ties by arrival order (`tie_policy='stable'`, exactly what Python's stable
`sorted(..., reverse=True)` does) or by canonical key, larger first (`tie_policy='det'`).
"""
from bisect import insort
from collections.abc import Callable

import numpy as np
import torch

from .cardparser import CardIndices, get_deck
from .color import COLOR_NUM
from .engine import M64, Engine, heuristic_id, pack_aux, pack_key, unpack_record, _i64
from .gems import MAX_GEMS, Gems, increase_bonus, subtract_with_bonus

deck = get_deck()

#: most games in one State.solve_many batch (spl_sbatch_create's limit)
MAX_BATCH_GAMES = 1 << 16

#: module-level policy defaults (overridable per solve() call)
DEFAULT_TIE_POLICY = 'stable'
DEFAULT_NOISE = 'const'
DEFAULT_DEVICE = 0


def _engine(device=None) -> Engine:
    """The context solve()/__iter__/HEURISTICS run on.  Under torch.distributed (one process per GPU) the
    default is this rank's own GPU -- LOCAL_RANK, or torch's current device once the launcher has set it --
    never cuda:0 on every rank: NCCL cannot run two ranks on one device."""
    if device is None:
        device = DEFAULT_DEVICE
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            import os
            device = int(os.environ['LOCAL_RANK']) if 'LOCAL_RANK' in os.environ else torch.cuda.current_device()
            if torch.cuda.device_count() and device >= torch.cuda.device_count():
                raise RuntimeError(f'rank {dist.get_rank()} maps to cuda:{device}, but only {torch.cuda.device_count()} '
                                   f'devices are visible: run one process per GPU')
    return Engine.get(device)


def _score_one(name: str, state: 'State') -> float:
    eng = _engine()
    k = pack_key(state.cards, state.gems)
    keys = torch.tensor([[_i64(k), _i64(k >> 64)]], dtype=torch.int64, device=eng.tdev)
    aux = torch.tensor([_i64(pack_aux(state.bonus, state.pts, state.saved))], dtype=torch.int64, device=eng.tdev)
    return float(eng.score(name, keys, aux, DEFAULT_NOISE).item())


HeuristicFunc = Callable[['State'], float]


def simple_heuristic(state: 'State') -> float:
    """(saved**0.4)*(pts**2.5) + noise (src/solver.py:210-215), evaluated by spl_score."""
    return _score_one('simple', state)


def balanced_heuristic(state: 'State') -> float:
    """src/solver.py:218-249, evaluated by spl_score."""
    return _score_one('balanced', state)


def aggressive_heuristic(state: 'State') -> float:
    """src/solver.py:252-262, evaluated by spl_score."""
    return _score_one('aggressive', state)


def efficiency_heuristic(state: 'State') -> float:
    """src/solver.py:265-286, evaluated by spl_score."""
    return _score_one('efficiency', state)


def competitive_heuristic(state: 'State') -> float:
    """Alias of balanced for single-player states (src/solver.py:289-296)."""
    return balanced_heuristic(state)


HEURISTICS: dict[str, HeuristicFunc] = {
    'simple': simple_heuristic,
    'balanced': balanced_heuristic,
    'aggressive': aggressive_heuristic,
    'efficiency': efficiency_heuristic,
    'competitive': competitive_heuristic,
}


class State:
    """One player's position: cards, bonus, gems, pts, saved (src/solver.py:308-318)."""

    def __init__(self, cards, bonus, gems, pts, saved):
        self.cards: CardIndices = cards
        self.bonus: Gems = bonus
        self.gems: Gems = gems
        self.pts: int = pts
        self.saved: int = saved
        self.hash: int = hash((self.cards, self.gems))

    @classmethod
    def newgame(cls) -> 'State':
        z = (0,) * COLOR_NUM
        return State(cards=(), bonus=z, gems=z, pts=0, saved=0)

    @classmethod
    def from_record(cls, lo: int, hi: int, aux: int) -> 'State':
        cards, bonus, gems, pts, saved = unpack_record(lo, hi, aux)
        return State(cards=cards, bonus=bonus, gems=gems, pts=pts, saved=saved)

    def record(self) -> tuple[int, int]:
        """(128-bit key, 64-bit aux) of this state in the library's packed layout."""
        return pack_key(self.cards, self.gems), pack_aux(self.bonus, self.pts, self.saved)

    def __repr__(self):
        if self.cards:
            return f'{self.gems!r} {"-".join(str(deck[c]) for c in self.cards)}'
        return f'{self.gems!r}'

    def __hash__(self):
        return self.hash

    def __eq__(self, other) -> bool:
        return self.hash == other.hash

    def buy_card(self, card_num: int) -> 'State':
        """Buy without an affordability check, as src/solver.py:338-355 (host-side API mirror)."""
        cards_mut = list(self.cards)
        insort(cards_mut, card_num)
        card = deck[card_num]
        gems, saved = subtract_with_bonus(self.gems, card.cost, self.bonus)
        return State(cards=tuple(cards_mut), bonus=increase_bonus(self.bonus, card.bonus), gems=gems,
                     pts=self.pts + card.pt, saved=self.saved + saved)

    def __iter__(self):
        """Successors in reference order -- buys (ascending card index) then gem takes
        (src/solver.py:357-388) -- produced by the expand kernel."""
        yield from self._successors(_engine())

    def _successors(self, eng: Engine):
        k, a = self.record()
        keys = torch.tensor([[_i64(k), _i64(k >> 64)]], dtype=torch.int64, device=eng.tdev)
        aux = torch.tensor([_i64(a)], dtype=torch.int64, device=eng.tdev)
        ck, ca, _ = eng.expand(keys, aux)
        ck = ck.cpu().numpy().view(np.uint64)
        ca = ca.cpu().numpy().view(np.uint64)
        eng.host_bytes[0] += 24                  # the state's key + aux up ...
        eng.host_bytes[1] += ck.nbytes + ca.nbytes  # ... its successor list down
        return [State.from_record(int(ck[i, 0]), int(ck[i, 1]), int(ca[i])) for i in range(len(ca))]

    def solve(
        self,
        goal_pts: int = 15,
        *,
        use_heuristic: bool = False,
        heuristic_name: str = 'simple',
        beam_width: int = 300_000,
        verbose: bool = True,
        tie_policy: str | None = None,
        noise: str | None = None,
        device: int | None = None,
        engine: Engine | None = None,
        stats: list | None = None,
        identity: str = 'key',
    ) -> list['State']:
        """BFS / beam search on the GPU; same arguments and return value as src/solver.py:390-464.

        Extra keyword-only arguments (all optional): `tie_policy` ('stable' | 'det'), `noise`
        ('const' | 'hash' | 'mt'), `device`, `engine` (a pre-built Engine, e.g. with a larger visited
        table), `stats` (a list that receives one dict of counters per level) and `identity`
        ('key' = exact (cards, gems); 'pyhash' = dedup on the reference's own 64-bit
        hash((cards, gems)), src/solver.py:316, so that even hash collisions merge as they do there;
        single GPU only).
        """
        tie_policy = tie_policy or DEFAULT_TIE_POLICY
        noise = noise or DEFAULT_NOISE
        eng = engine or _engine(device)
        if verbose:
            print('=' * 60)
            print('SPEEDRUN MODE SOLVER')
            print('=' * 60)
            print(f'Target Points: {goal_pts}')
            print(f'Heuristic: {heuristic_name if use_heuristic else "None (pure BFS)"}')
            if use_heuristic:
                print(f'Beam Width: {beam_width:,}')
            print('Gem Pool: Infinite')
            print('Card Visibility: All 90 cards')
            print('=' * 60)
            print()
        k, a = self.record()
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            # one process per GPU (torchrun): every rank calls solve() collectively; the frontier is
            # sharded by key hash and each level is bit-identical to the single-GPU search
            from .sharded import Comm, CudaBackend, DictionaryOverflow, GroupedShardedSolver, ShardedSolver

            def key_sharded():  # exhaustive BFS, key ties, hash / mt noise, pyhash identity: queue sharded by key hash
                return ShardedSolver(CudaBackend(eng), Comm(eng.tdev), k, a, goal_pts, use_heuristic, heuristic_name,
                                     beam_width, tie_policy, noise, identity=identity)

            def run(sh):
                try:
                    infos = list(sh.run())
                    return infos, sh.path()[1]
                finally:
                    if hasattr(sh, 'close'):
                        sh.close()
            if use_heuristic and tie_policy == 'stable' and noise == 'const' and identity == 'key':
                # queue sharded by card set: gem takes never leave the GPU, only card buys are routed
                sh = GroupedShardedSolver(eng, Comm(eng.tdev), k, a, goal_pts, heuristic_name, beam_width, noise)
                try:
                    infos, ordinals = run(sh)
                except DictionaryOverflow:  # too many distinct scores for the dictionary cut (every rank gets here together)
                    sh = key_sharded()
                    infos, ordinals = run(sh)
            else:
                sh = key_sharded()
                infos, ordinals = run(sh)
            if stats is not None:
                stats.extend(infos)
            if sh.noise_source is not None:
                sh.noise_source.finish()
            path = [self]
            for o in ordinals:
                path.append(path[-1]._successors(eng)[o])
            return path
        sol = eng.solver(k, a, goal_pts, use_heuristic, heuristic_name, beam_width, tie_policy, noise, identity=identity)
        try:
            turn = 0
            max_pts = 0
            while True:
                if verbose:
                    max_pts = _print_progress(sol, turn, max_pts, goal_pts)
                info = sol.step()
                if stats is not None:
                    stats.append(info)
                turn += 1
                if info['ended']:
                    break
            _, ordinals = sol.path()
            if sol.noise_source is not None:
                sol.noise_source.finish()  # leave `random` where the reference's own solve() would
        finally:
            sol.close()
        # replay the winning line through __iter__ so every field (saved, bonus, pts) is exact
        path = [self]
        for o in ordinals:
            path.append(path[-1]._successors(eng)[o])
        return path

    @classmethod
    def solve_many(
        cls,
        roots,
        goal_pts=15,
        *,
        use_heuristic=False,
        heuristic_name='simple',
        beam_width=300_000,
        tie_policy: str | None = None,
        noise: str | None = None,
        device: int | None = None,
        engine: Engine | None = None,
        stats: list | None = None,
    ) -> list[list['State']]:
        """`root.solve(goal_pts=..., use_heuristic=..., heuristic_name=..., beam_width=..., tie_policy=..., noise=...,
        verbose=False)` for every root of `roots`, searched together on one GPU: the games advance one level at a time
        in lockstep, and each returns exactly the line its own solve() returns.

        `goal_pts`, `use_heuristic`, `heuristic_name` and `beam_width` are one value or one per root; `tie_policy`
        ('stable' | 'det') and `noise` ('const' | 'hash': 'mt' draws would depend on the other games) hold for the
        whole batch.  Equal roots are separate games.  Nothing is printed.  With `stats`, one dict per level is
        appended: the aggregate counters and 'games', the per-game counters.  Every argument is checked before the
        GPU is used."""
        roots = list(roots)
        if not roots:
            raise ValueError('solve_many needs at least one root')
        n = len(roots)
        if n > MAX_BATCH_GAMES:
            raise ValueError(f'solve_many: {n} roots, at most {MAX_BATCH_GAMES} in one batch')

        def per_game(value, name):
            if np.ndim(value) == 0:  # one value (str, int, bool, numpy scalar) for every root
                return [value] * n
            values = list(value)
            if len(values) != n:
                raise ValueError(f'solve_many: {len(values)} values of {name} for {n} roots')
            return values

        goals = [int(g) for g in per_game(goal_pts, 'goal_pts')]
        kinds = [bool(u) for u in per_game(use_heuristic, 'use_heuristic')]
        names = per_game(heuristic_name, 'heuristic_name')
        beams = [int(b) for b in per_game(beam_width, 'beam_width')]
        if any(b < 1 for b in beams):
            raise ValueError('solve_many: every beam width must be >= 1')
        tie_policy = tie_policy or DEFAULT_TIE_POLICY
        noise = noise or DEFAULT_NOISE
        if tie_policy not in ('stable', 'det'):
            raise ValueError(f"solve_many supports tie_policy 'stable' and 'det', not {tie_policy!r}")
        if noise not in ('const', 'hash'):
            raise ValueError(f"solve_many supports noise 'const' and 'hash', not {noise!r}: 'mt' draws depend on the other games")
        rows = np.zeros((n, 4), np.uint64)
        for g, r in enumerate(roots):
            if len(r.gems) != COLOR_NUM or any(not 0 <= x <= MAX_GEMS for x in r.gems) or sum(r.gems) > 10:
                raise ValueError(f'solve_many: root {g} has an illegal gem hand {r.gems!r}')
            if any(not 0 <= c < len(deck) for c in r.cards):
                raise ValueError(f'solve_many: root {g} holds a card index outside 0..{len(deck) - 1}')
            k, a = r.record()
            rows[g] = (k & M64, k >> 64, a, M64)
        eng = engine or _engine(device)
        sol = eng.sbatch_solver(rows, goals, kinds, [heuristic_id(h) for h in names], beams, tie_policy, noise)
        try:
            while not sol.ended:
                info = sol.step()
                if stats is not None:
                    stats.append(info)
            lines = sol.lines()
        finally:
            sol.close()
        return [[root] + [State.from_record(int(lo), int(hi), int(aux)) for lo, hi, aux, _ in line[1:]]
                for root, line in zip(roots, lines)]


def _print_progress(sol, turn: int, max_pts: int, goal_pts: int) -> int:
    """The reference's verbose lines (src/solver.py:436-442): queue head, then every state that
    raises the running maximum of pts while the queue is scanned (up to the goal state)."""
    fr = sol.frontier()
    n = fr.shape[0]
    if n == 0:
        return max_pts
    head = fr[0].cpu().numpy().view(np.uint64)
    print(f'{turn=:<10} {State.from_record(int(head[0]), int(head[1]), int(head[2]))}')
    pts = (fr[:, 2] >> 16) & 0xff
    goal_hits = torch.nonzero(pts >= goal_pts)
    stop = int(goal_hits[0]) + 1 if goal_hits.numel() else n
    run = torch.cummax(pts[:stop], 0).values
    prev = torch.cat([torch.full((1,), max_pts, dtype=run.dtype, device=run.device), run[:-1]])
    prev = torch.clamp(prev, min=max_pts)
    for i in torch.nonzero(pts[:stop] > prev).flatten().tolist():
        rec = fr[i].cpu().numpy().view(np.uint64)
        st = State.from_record(int(rec[0]), int(rec[1]), int(rec[2]))
        max_pts = st.pts
        print(f'{max_pts=:<7} {st}')
    return max_pts
