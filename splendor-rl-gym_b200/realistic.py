"""Realistic multi-player mode: the reference's GameConfig / GemPool / CardMarket / PlayerState /
MultiPlayerState surface (src/solver.py:25-200, 471-860) driven by the CUDA library.

`MultiPlayerState.solve()` -> spl_rsolver_* (with `shard=True`: RShardedSolver over the ranks of the process group,
sharded.py) ; `solve_many()` -> spl_rbatch_* (many games in lockstep on one GPU) ; `__iter__` -> spl_rexpand on one record; the
competitive heuristic -> spl_rscore.  The card market order (optionally shuffled with Python's
`random.Random(seed)` exactly as CardMarket.from_full_deck does) is computed here on the host and
handed to the kernels as an input table.  The reference draws tie-break noise from the unseeded
global RNG; here `randint` is the declared constant 50 (`noise='const'`) and score ties fall to
arrival order, which is what the reference's stable `sorted(..., reverse=True)` does.
"""
import ctypes as C
import numbers
import random
from dataclasses import dataclass

import numpy as np
import torch

from ._lib import check, lib
from .cardparser import CardIndices, get_deck
from .color import COLOR_NUM
from .engine import NOISE_IDS, Engine, LevelInfo, _DevArray
from .gems import Gems

deck = get_deck()

RPLAYER_DTYPE = np.dtype([('mlo', '<u8'), ('mhi', '<u4'), ('gems', '<u2'), ('saved', '<u2')])
RREC_DTYPE = np.dtype([('p', RPLAYER_DTYPE, (4,)), ('vis', 'u1', (12,)), ('cur', 'u1'), ('pad', 'u1', (3,)),
                       ('link', '<u8'), ('spare', '<u8')])


class RConfig(C.Structure):
    _fields_ = [('num_players', C.c_int32), ('target_points', C.c_int32), ('gems_per_color', C.c_int32),
                ('noise', C.c_int32), ('deck_len', C.c_int32 * 3), ('deck', (C.c_uint8 * 40) * 3)]


@dataclass(frozen=True)
class GameConfig:
    """Game rules (src/solver.py:25-33)."""
    num_players: int = 2
    target_points: int = 15
    gems_per_color: int = 4  # 4 for 2p, 5 for 3p, 7 for 4p
    cards_visible_per_tier: int = 4
    infinite_resources: bool = True


@dataclass(frozen=True)
class GemPool:
    """Gem pool of the table (src/solver.py:36-80)."""
    available: Gems

    @classmethod
    def new_pool(cls, gems_per_color: int) -> 'GemPool':
        return cls(available=tuple(gems_per_color for _ in range(COLOR_NUM)))

    def can_take_three_different(self, gems_requested: Gems) -> bool:
        if sum(1 for g in gems_requested if g > 0) != 3:
            return False
        return all(gems_requested[i] <= 1 and self.available[i] >= gems_requested[i] for i in range(COLOR_NUM))

    def can_take_two_same(self, gems_requested: Gems) -> bool:
        if sum(gems_requested) != 2:
            return False
        idx = next((i for i in range(COLOR_NUM) if gems_requested[i] == 2), None)
        return idx is not None and self.available[idx] >= 4

    def take(self, gems: Gems) -> 'GemPool':
        return GemPool(tuple(a - g for a, g in zip(self.available, gems)))

    def return_gems(self, gems: Gems) -> 'GemPool':
        return GemPool(tuple(a + g for a, g in zip(self.available, gems)))


@dataclass(frozen=True)
class CardMarket:
    """Visible cards and remaining decks per tier (src/solver.py:83-174)."""
    tier1_visible: tuple[int, ...]
    tier2_visible: tuple[int, ...]
    tier3_visible: tuple[int, ...]
    tier1_deck: tuple[int, ...]
    tier2_deck: tuple[int, ...]
    tier3_deck: tuple[int, ...]

    @classmethod
    def from_full_deck(cls, shuffle: bool = False, seed: int | None = None) -> 'CardMarket':
        tiers = [[i for i, c in enumerate(deck) if c.pt == 0], [i for i, c in enumerate(deck) if c.pt in (1, 2)],
                 [i for i, c in enumerate(deck) if c.pt >= 3]]  # tiers by points, :102-104
        if shuffle:
            rng = random.Random(seed)
            for t in tiers:
                rng.shuffle(t)
        return cls(tuple(tiers[0][:4]), tuple(tiers[1][:4]), tuple(tiers[2][:4]),
                   tuple(tiers[0][4:]), tuple(tiers[1][4:]), tuple(tiers[2][4:]))

    def buy_card(self, card_idx: int) -> 'CardMarket':
        vis = [list(self.tier1_visible), list(self.tier2_visible), list(self.tier3_visible)]
        dk = [self.tier1_deck, self.tier2_deck, self.tier3_deck]
        for t in range(3):
            if card_idx in vis[t]:
                vis[t].remove(card_idx)
                if dk[t]:
                    vis[t].append(dk[t][0])
                    dk[t] = dk[t][1:]
                return CardMarket(tuple(vis[0]), tuple(vis[1]), tuple(vis[2]), dk[0], dk[1], dk[2])
        return self

    def all_visible_cards(self) -> tuple[int, ...]:
        return self.tier1_visible + self.tier2_visible + self.tier3_visible


@dataclass(frozen=True)
class PlayerState:
    """One player (src/solver.py:177-200)."""
    player_id: int
    cards: CardIndices
    bonus: Gems
    gems: Gems
    pts: int
    saved: int

    def total_gem_count(self) -> int:
        return sum(self.gems)

    def can_afford(self, card_idx: int) -> bool:
        cost = deck[card_idx].cost
        return all(self.gems[i] + self.bonus[i] >= cost[i] for i in range(COLOR_NUM))


def _tier_of(card: int) -> int:
    pt = deck[card].pt
    return 0 if pt == 0 else 1 if pt <= 2 else 2


class MultiPlayerState:
    """Complete game state of realistic mode (src/solver.py:471-566)."""

    def __init__(self, config: GameConfig, players, gem_pool: GemPool, market: CardMarket, current_player: int,
                 turn_number: int, final_round_triggered: bool = False, final_round_player: int | None = None,
                 _sequences=None):
        self.config = config
        self.players = players
        self.gem_pool = gem_pool
        self.market = market
        self.current_player = current_player
        self.turn_number = turn_number
        self.final_round_triggered = final_round_triggered
        self.final_round_player = final_round_player
        self.hash = hash((self.players, self.gem_pool.available, self.market.all_visible_cards(), self.current_player))
        # full tier sequences (cards ever visible or still in the deck, in draw order): kernel input table
        self._sequences = _sequences or self._derive_sequences()

    def _derive_sequences(self):
        owned = sorted(c for p in self.players for c in p.cards)
        seqs = []
        for t, (vis, dk) in enumerate(((self.market.tier1_visible, self.market.tier1_deck),
                                       (self.market.tier2_visible, self.market.tier2_deck),
                                       (self.market.tier3_visible, self.market.tier3_deck))):
            # bought cards precede everything still on the table in draw order; their relative order is irrelevant
            seqs.append(tuple([c for c in owned if _tier_of(c) == t] + list(vis) + list(dk)))
        return tuple(seqs)

    @classmethod
    def newgame(cls, config: GameConfig | None = None, shuffle_market: bool = False, seed: int | None = None):
        if config is None:
            config = GameConfig(infinite_resources=False)
        z = (0,) * COLOR_NUM
        players = tuple(PlayerState(player_id=i, cards=(), bonus=z, gems=z, pts=0, saved=0)
                        for i in range(config.num_players))
        return cls(config=config, players=players, gem_pool=GemPool.new_pool(config.gems_per_color),
                   market=CardMarket.from_full_deck(shuffle_market, seed), current_player=0, turn_number=0)

    def __repr__(self):
        cur = self.players[self.current_player]
        return f'Turn {self.turn_number}, P{self.current_player}: {cur.pts}pts, {cur.gems!r}'

    def __hash__(self):
        return self.hash

    def __eq__(self, other) -> bool:
        return self.hash == other.hash

    def is_game_over(self) -> bool:
        if not self.final_round_triggered:
            return any(p.pts >= self.config.target_points for p in self.players)
        return self.current_player == self.final_round_player

    def get_winner(self) -> int | None:
        if not self.is_game_over():
            return None
        max_pts = max(p.pts for p in self.players)
        winners = [p for p in self.players if p.pts == max_pts]
        if len(winners) == 1:
            return winners[0].player_id
        min_cards = min(len(p.cards) for p in winners)
        winners = [p for p in winners if len(p.cards) == min_cards]
        return winners[0].player_id if len(winners) == 1 else None

    # ---------------------------------------------------------------- packing
    def rconfig(self, noise: str = 'const') -> RConfig:
        if self.config.infinite_resources:
            raise NotImplementedError('MultiPlayerState with infinite_resources=True is the speedrun rule set; use State')
        cfg = RConfig(self.config.num_players, self.config.target_points, self.config.gems_per_color, NOISE_IDS[noise])
        for t, seq in enumerate(self._sequences):
            cfg.deck_len[t] = len(seq)
            for i, c in enumerate(seq):
                cfg.deck[t][i] = c
        return cfg

    def record(self) -> np.ndarray:
        rec = np.zeros(1, RREC_DTYPE)
        for i, p in enumerate(self.players):
            m = 0
            for c in p.cards:
                m |= 1 << c
            g = 0
            for k, x in enumerate(p.gems):
                g |= x << (3 * k)
            rec['p'][0][i] = (m & ((1 << 64) - 1), m >> 64, g, p.saved)
        vis = []
        for tier in (self.market.tier1_visible, self.market.tier2_visible, self.market.tier3_visible):
            vis += list(tier) + [255] * (4 - len(tier))
        rec['vis'][0] = vis
        rec['cur'] = self.current_player
        rec['link'] = (1 << 64) - 1
        return rec

    def _child_from_record(self, rec) -> 'MultiPlayerState':
        cfg = self.config
        players = []
        for i in range(cfg.num_players):
            m = int(rec['p'][i]['mlo']) | int(rec['p'][i]['mhi']) << 64
            cards = tuple(c for c in range(90) if (m >> c) & 1)
            bonus = [0] * COLOR_NUM
            for c in cards:
                bonus[deck[c].bonus.value] += 1
            g = int(rec['p'][i]['gems'])
            players.append(PlayerState(player_id=i, cards=cards, bonus=tuple(bonus),
                                       gems=tuple((g >> (3 * k)) & 7 for k in range(COLOR_NUM)),
                                       pts=sum(deck[c].pt for c in cards), saved=int(rec['p'][i]['saved'])))
        pool = tuple(cfg.gems_per_color - sum(p.gems[k] for p in players) for k in range(COLOR_NUM))
        vis = [[int(v) for v in rec['vis'][4 * t:4 * t + 4] if v != 255] for t in range(3)]
        owned = {c for p in players for c in p.cards}
        decks = []
        for t in range(3):
            seq = self._sequences[t]
            n_owned = sum(1 for c in owned if _tier_of(c) == t)
            decks.append(tuple(seq[4 + n_owned:]))
        market = CardMarket(tuple(vis[0]), tuple(vis[1]), tuple(vis[2]), decks[0], decks[1], decks[2])
        mover = players[self.current_player]
        triggered = self.final_round_triggered or mover.pts >= cfg.target_points        # :607-610
        frp = (self.final_round_player if self.final_round_triggered
               else self.current_player if triggered else None)                          # :611-615
        return MultiPlayerState(cfg, tuple(players), GemPool(pool), market, int(rec['cur']), self.turn_number + 1,
                                triggered, frp, _sequences=self._sequences)

    @staticmethod
    def _rec_pts(rec, player: int) -> int:
        m = int(rec['p'][player]['mlo']) | int(rec['p'][player]['mhi']) << 64
        return sum(deck[c].pt for c in range(90) if (m >> c) & 1)

    def _successors(self, eng: Engine, noise='const'):
        recs = eng.rexpand(self.rconfig(noise), self.record())
        return [self._child_from_record(r) for r in recs]

    def __iter__(self):
        """Successors in reference order (src/solver.py:568-748), produced by spl_rexpand."""
        from .solver import _engine
        yield from self._successors(_engine())

    def heuristic(self, noise: str = 'const') -> float:
        """multi_competitive_heuristic (src/solver.py:778-812) of this state, via spl_rscore."""
        from .solver import _engine
        return float(_engine().rscore(self.rconfig(noise), self.record())[0])

    def solve(self, *, use_heuristic: bool = True, heuristic_name: str = 'competitive', beam_width: int = 20_000,
              verbose: bool = True, noise: str = 'const', device: int | None = None, engine: Engine | None = None,
              stats: list | None = None, shard: bool = False) -> list['MultiPlayerState']:
        """Beam search over the multi-player game; arguments and return value as src/solver.py:750-860
        (`use_heuristic` / `heuristic_name` are ignored there too: the beam is always applied).

        Without `shard`, every process solves the whole game on its own GPU (under torchrun: one replica per rank).
        `shard=True` spreads one search over the ranks of the default process group (a world of 1 when none is
        initialised): every rank calls solve() collectively, each holds a slice of the queue and of the visited set,
        so a beam too wide for one GPU's visited table can run, and every level equals the single-GPU search.  It
        supports noise 'const' and 'hash' ('mt' raises ValueError).  With `verbose`, rank 0 prints the banner and the
        `turn=... Queue size:` lines; the `max_pts=` progress lines are not printed on the sharded path."""
        from .solver import _engine
        if shard and noise == 'mt':
            raise ValueError("solve(shard=True) supports noise 'const' and 'hash', not 'mt'")
        eng = engine or _engine(device)
        if shard:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized() and dist.get_rank() != 0:
                verbose = False
        if verbose:
            print('=' * 60)
            print('REALISTIC MODE SOLVER')
            print('=' * 60)
            print(f'Target Points: {self.config.target_points}')
            print(f'Number of Players: {self.config.num_players}')
            print(f'Gems per Color: {self.config.gems_per_color}')
            print(f'Heuristic: {heuristic_name}')
            print(f'Beam Width: {beam_width:,}')
            print('Card Visibility: 12 cards (4 per tier)')
            print(f'Market Shuffled: {"Yes" if self.market.tier1_deck != self.market.tier1_deck[:1] else "No (deterministic)"}')
            print('=' * 60)
            print()
        rcfg = self.rconfig(noise)
        if shard:
            ordinals = self._solve_sharded(eng, rcfg, beam_width, verbose, stats)
        else:
            ordinals = self._solve_local(eng, rcfg, beam_width, verbose, stats)
        path = [self]
        for o in ordinals:
            path.append(path[-1]._successors(eng, noise)[o])
        return path

    def _solve_sharded(self, eng: Engine, rcfg: RConfig, beam_width: int, verbose: bool, stats) -> list[int]:
        from .sharded import Comm, RCudaBackend, RShardedSolver
        comm = Comm(eng.tdev)
        sol = RShardedSolver(RCudaBackend(eng, rcfg, self.record()), comm, beam_width)
        turn = 0
        while True:
            if verbose and turn % 100 == 0:
                print(f'{turn=:<10} Queue size: {sol.N}')
            info = sol.step()
            if stats is not None:
                stats.append(info)
            turn += 1
            if info['ended']:
                break
        if turn > 1000 and comm.rank == 0:
            print('Warning: Reached turn limit (1000)')
        return sol.path()[1]

    def _solve_local(self, eng: Engine, rcfg: RConfig, beam_width: int, verbose: bool, stats) -> list[int]:
        sol = eng.rsolver(rcfg, self.record(), beam_width)
        try:
            turn = 0
            max_pts = 0
            while True:
                if verbose and turn % 100 == 0:
                    print(f'{turn=:<10} Queue size: {sol.frontier_size()}')
                if verbose:  # `max_pts=...` lines of src/solver.py:832-836 (states before the first finished game)
                    for _, rec, mp in sol.progress(rcfg, max_pts):
                        cur = int(rec['cur'])
                        if self._rec_pts(rec, cur) >= self.config.target_points:
                            break
                        max_pts = mp
                        g = int(rec['p'][cur]['gems'])
                        gems = tuple((g >> (3 * k)) & 7 for k in range(COLOR_NUM))
                        print(f'{max_pts=:<7} Turn {turn}, P{cur}: {self._rec_pts(rec, cur)}pts, {gems!r}')
                info = sol.step()
                if stats is not None:
                    stats.append(info)
                turn += 1
                if info['ended']:
                    break
            if turn > 1000:
                print('Warning: Reached turn limit (1000)')
            _, ordinals = sol.path()
            if sol.noise_source is not None:
                sol.noise_source.finish()
        finally:
            sol.close()
        return ordinals


def solve_many(roots, *, beam_width=20_000, noise: str = 'const', device: int | None = None, engine: Engine | None = None,
               stats: list | None = None) -> list[list[MultiPlayerState]]:
    """`root.solve(beam_width=..., noise=..., verbose=False)` for every root of `roots`, searched together on one GPU:
    the games advance one level at a time in lockstep, each with its own rules, market and beam width (`beam_width` is
    one int or one per game), and each returns exactly the line its own solve() returns.  noise is 'const' or 'hash'
    ('mt' draws depend on the other games).  With `stats`, one dict per level is appended: the aggregate counters and
    'games', the per-game counters."""
    from .solver import MAX_BATCH_GAMES, _engine
    roots = list(roots)
    if not roots:
        raise ValueError('solve_many needs at least one game')
    if len(roots) > MAX_BATCH_GAMES:
        raise ValueError(f'solve_many: {len(roots)} roots, at most {MAX_BATCH_GAMES} in one batch')
    for r in roots:
        if r.config.infinite_resources:
            raise ValueError('solve_many: a root with infinite_resources=True follows the speedrun rules; use State.solve')
    if noise not in ('const', 'hash'):
        raise ValueError(f"solve_many supports noise 'const' and 'hash', not {noise!r}: 'mt' draws depend on the other games")
    beams = [beam_width] * len(roots) if isinstance(beam_width, numbers.Integral) else list(beam_width)
    if len(beams) != len(roots):
        raise ValueError(f'solve_many: {len(beams)} beam widths for {len(roots)} games')
    if any(int(b) < 1 for b in beams):
        raise ValueError('solve_many: every beam width must be >= 1')
    eng = engine or _engine(device)
    sol = eng.rbatch_solver([r.rconfig(noise) for r in roots], np.concatenate([r.record() for r in roots]),
                            [int(b) for b in beams])
    try:
        while not sol.ended:
            info = sol.step()
            if stats is not None:
                stats.append(info)
        lines = sol.lines()
    finally:
        sol.close()
    out = []
    for root, recs in zip(roots, lines):
        path = [root]
        for rec in recs[1:]:
            path.append(path[-1]._child_from_record(rec))
        out.append(path)
    return out
